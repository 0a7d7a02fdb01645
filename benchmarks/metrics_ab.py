"""Times b200dct_roundtrip_metrics at 8192^2 (f32 and u8, default plan) for one or more builds of
libb200dct.so, alternating between them round by round so that every build sees the same machine state.

    python benchmarks/metrics_ab.py [--rounds 5] [--iters 200] LIB [LIB ...]

Inputs rotate over three images (768 MiB of f32 pixels in, as much out: far more than L2).  Prints one
JSON line per (library, dtype) with the median and spread of the per-round means in microseconds, and
the GPU's name and power limit."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess

import torch


def load(path):
    L = C.CDLL(path)
    vp, sz, i = C.c_void_p, C.c_size_t, C.c_int
    L.b200dct_plan_create.argtypes = [C.POINTER(vp)]
    L.b200dct_metrics_workspace_bytes.argtypes = [i, i]
    L.b200dct_metrics_workspace_bytes.restype = sz
    L.b200dct_roundtrip_metrics.argtypes = [vp, vp, i, sz, vp, i, sz, vp, i, sz, i, i, vp, vp, sz, vp]
    plan = vp()
    assert L.b200dct_plan_create(C.byref(plan)) == 0
    return L, plan


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs="+")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--n", type=int, default=8192)
    a = ap.parse_args()
    N = a.n
    stream = torch.cuda.Stream()
    sp = C.c_void_p(stream.cuda_stream)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    libs = [load(p) for p in a.libs]
    res = {}
    for code, dt, es in ((0, torch.float32, 4), (1, torch.uint8, 1)):
        xs = [torch.randint(0, 256, (N, N), device="cuda", dtype=torch.int32).to(dt) for _ in range(3)]
        ys = [torch.empty_like(x) for x in xs]
        acc = torch.zeros(3, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        for r in range(a.rounds + 1):                 # round 0 warms up every build
            for li, (L, plan) in enumerate(libs):
                nb = int(L.b200dct_metrics_workspace_bytes(N, N))
                ws = torch.empty(max(1, nb // 8), dtype=torch.float64, device="cuda")
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for i in range(a.iters):
                    rc = L.b200dct_roundtrip_metrics(plan, xs[i % 3].data_ptr(), code, N * es, ys[i % 3].data_ptr(), code,
                                                     N * es, None, 0, 0, N, N, acc.data_ptr(), ws.data_ptr(), nb, sp)
                    assert rc == 0, rc
                e1.record(stream)
                e1.synchronize()
                if r:
                    res.setdefault((a.libs[li], str(dt)), []).append(e0.elapsed_time(e1) * 1000.0 / a.iters)
        del xs, ys
    for (lib, dt), v in res.items():
        v = sorted(v)
        print(json.dumps({"lib": lib, "dtype": dt, "N": N, "us_median": round(v[len(v) // 2], 2),
                          "us_min": round(v[0], 2), "us_max": round(v[-1], 2), "rounds": v and len(v), "gpu": gpu}))


if __name__ == "__main__":
    main()
