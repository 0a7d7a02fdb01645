"""Retained-coefficient round trips (k = 6..10, all): u8 and f32 at N^2, AUTO path."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
import cuda_dct_idct_b200 as m
N = int(os.environ.get("N", 8192)); iters = int(os.environ.get("ITERS", 200))
dev = torch.device("cuda")
def t(fn):
    for i in range(5): fn(i)
    torch.cuda.synchronize(); best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters): fn(i)
        e1.record(); torch.cuda.synchronize(); best = min(best, e0.elapsed_time(e1) / iters)
    return best
for name, dt, paths in (("u8", torch.uint8, (0, 2)), ("f32", torch.float32, (0, 1))):
    ins = [torch.randint(0, 256, (N, N), device=dev, dtype=torch.int32).to(dt) for _ in range(4)]
    outs = [torch.empty_like(x) for x in ins]
    for path in paths:
        for k in (6, 7, 8, 9, 10, 64):
            plan = m.Plan(keep=m.zigzag_mask(k), path=path)
            ms = t(lambda i: m.roundtrip(ins[i % 4], out=outs[i % 4], plan=plan))
            print(f"{name} N={N} k={k:2d} {('auto','direct','tma')[path]:6s}->{m.api.last_path():6s} {ms*1e3:8.1f} us  {N*N/ms/1e6:8.1f} Gpx/s", flush=True)
