"""The 4:2:0 colour calls at 8192^2 RGB, us per call, next to the 4:4:4 split calls in the same run:
b200dct_forward_rgb420 / b200dct_inverse_rgb420 and the pair back to back against b200dct_forward_rgb /
b200dct_inverse_rgb and their pair.

Every variant alternates two sets of buffers (two 201 MB RGB inputs, two stream sets of 201 MB for 4:2:0 and 403 MB
for 4:4:4, two 201 MB outputs), so no call finds its input in the 126 MB L2.  The 4:2:0 and 4:4:4 variants
alternate window by window, so both share the box and the clock.  CUDA events around --iters back-to-back calls
after a warm-up, --reps windows per variant, the median window reported with the spread.  Bytes are what the
algorithm moves (4:2:0: forward 3 B/px read + 3 B/px streams written, inverse 3 + 3; 4:4:4: 3 + 6 and 6 + 3); the
share of peak is against the project's measured HBM copy peak (DESIGN.md section 4).

    python benchmarks/rgb420.py [--n 8192] [--iters 200] [--reps 7] [--out FILE]
"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import cuda_dct_idct_b200 as m  # noqa: E402

COPY_PEAK_GBS = 6538.6  # DESIGN.md section 4: measured HBM copy peak of a B200, GB/s


def window(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rgb420.py needs a CUDA device")
    N = a.n
    px = N * N
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    g = torch.Generator(device="cuda").manual_seed(3)
    rgb = [torch.randint(0, 256, (N, N, 3), device="cuda", generator=g, dtype=torch.int32).to(torch.uint8) for _ in range(2)]
    out = [torch.empty_like(rgb[0]) for _ in range(2)]
    zz444 = [torch.empty((3, N // 8, N // 8, 64), dtype=torch.int16, device="cuda") for _ in range(2)]
    zz420 = [(torch.empty((N // 8, N // 8, 64), dtype=torch.int16, device="cuda"),
              torch.empty((N // 16, N // 16, 64), dtype=torch.int16, device="cuda"),
              torch.empty((N // 16, N // 16, 64), dtype=torch.int16, device="cuda")) for _ in range(2)]

    lines = [f"# b200dct colour split calls, 4:2:0 against 4:4:4, {N}^2 RGB ({3 * px / 1e6:.0f} MB per image), one GPU: {gpu}",
             f"# benchmarks/rgb420.py --n {N} --iters {a.iters} --reps {a.reps} --warmup {a.warmup}; two buffer sets alternate "
             f"(larger than L2); 4:2:0 and 4:4:4 windows alternate; us per call = median of {a.reps} windows of {a.iters} "
             "back-to-back calls [min, max]",
             f"# share of peak: algorithmic bytes / time against the measured HBM copy peak {COPY_PEAK_GBS} GB/s"]
    for mode, plan in (("default (factored inverse)", m.Plan()), ("exact inverse", m.Plan(inverse=m.api.INVERSE_EXACT))):
        def pair420(i):
            m.forward_rgb420(rgb[i % 2], streams=zz420[i % 2], plan=plan)
            m.inverse_rgb420(zz420[i % 2], out=out[i % 2], plan=plan)

        def pair444(i):
            m.forward_rgb(rgb[i % 2], streams=zz444[i % 2], plan=plan)
            m.inverse_rgb(zz444[i % 2], out=out[i % 2], plan=plan)

        variants = (
            (("forward_rgb420", 6, lambda i: m.forward_rgb420(rgb[i % 2], streams=zz420[i % 2], plan=plan)),
             ("forward_rgb", 9, lambda i: m.forward_rgb(rgb[i % 2], streams=zz444[i % 2], plan=plan))),
            (("inverse_rgb420", 6, lambda i: m.inverse_rgb420(zz420[i % 2], out=out[i % 2], plan=plan)),
             ("inverse_rgb", 9, lambda i: m.inverse_rgb(zz444[i % 2], out=out[i % 2], plan=plan))),
            (("forward_rgb420 + inverse_rgb420", 12, pair420), ("forward_rgb + inverse_rgb", 18, pair444)),
        )
        lines.append(f"## {mode}")
        for duo in variants:
            for _, _, fn in duo:
                for i in range(a.warmup):
                    fn(i)
            torch.cuda.synchronize()
            times = [[], []]
            for _ in range(a.reps):
                for k, (_, _, fn) in enumerate(duo):
                    times[k].append(window(fn, a.iters))
            for (name, bpp, _), t in zip(duo, times):
                us = statistics.median(t)
                gbs = bpp * px / us / 1e3
                lines.append(f"{name:40s} {us:8.1f} us [{min(t):.1f}, {max(t):.1f}]  {bpp:2d} B/px {gbs:7.1f} GB/s  "
                             f"{gbs / COPY_PEAK_GBS:.3f} of the copy peak")
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
