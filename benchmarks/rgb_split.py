"""The colour entry points at 8192^2 RGB, us per call: the fused round trip (b200dct_roundtrip_rgb, with and
without the coefficient streams) against its two halves (b200dct_forward_rgb, b200dct_inverse_rgb) and the
two halves back to back.

Every variant alternates two sets of buffers (two 201 MB RGB inputs, two 403 MB stream triples, two
201 MB outputs), so no call finds its input in the 126 MB L2.  CUDA events around --iters back-to-back
calls after a warm-up, --reps windows per variant, the median window reported with the spread.  Bytes are
what the algorithm moves (forward 3 B/px read + 6 B/px streams written, inverse 6 + 3, fused 3 + 3, + 6
with streams); the share of peak is against the project's measured HBM copy peak (DESIGN.md section 4),
and a plain device-to-device copy of an input is timed in the same run for comparison.

    python benchmarks/rgb_split.py [--n 8192] [--iters 200] [--reps 5] [--out FILE]
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


def time_window(fn, iters, reps, warmup):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    per_call = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        per_call.append(e0.elapsed_time(e1) * 1e3 / iters)
    return statistics.median(per_call), min(per_call), max(per_call)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rgb_split.py needs a CUDA device")
    N = a.n
    px = N * N
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    g = torch.Generator(device="cuda").manual_seed(3)
    rgb = [torch.randint(0, 256, (N, N, 3), device="cuda", generator=g, dtype=torch.int32).to(torch.uint8) for _ in range(2)]
    out = [torch.empty_like(rgb[0]) for _ in range(2)]
    zz = [torch.empty((3, N // 8, N // 8, 64), dtype=torch.int16, device="cuda") for _ in range(2)]
    copy_dst = torch.empty_like(rgb[0])

    lines = [f"# b200dct colour entry points, {N}^2 RGB ({3 * px / 1e6:.0f} MB per image), one GPU: {gpu}",
             f"# benchmarks/rgb_split.py --n {N} --iters {a.iters} --reps {a.reps} --warmup {a.warmup}; two buffer sets alternate "
             f"(larger than L2); us per call = median of {a.reps} windows of {a.iters} back-to-back calls [min, max]",
             f"# share of peak: algorithmic bytes / time against the measured HBM copy peak {COPY_PEAK_GBS} GB/s"]
    us, lo, hi = time_window(lambda i: copy_dst.copy_(rgb[i % 2]), a.iters, a.reps, a.warmup)
    lines.append(f"{'device-to-device copy of one input (torch copy_)':58s} {us:8.1f} us [{lo:.1f}, {hi:.1f}]   6 B/px "
                 f"{6 * px / us / 1e3:7.1f} GB/s  {6 * px / us / 1e3 / COPY_PEAK_GBS:.3f} of the copy peak")
    for mode, plan in (("default (factored inverse)", m.Plan()), ("exact inverse", m.Plan(inverse=m.api.INVERSE_EXACT))):
        # the split reproduces the fused call at this size before anything is timed
        ref_zz = torch.empty_like(zz[0])
        ref = m.roundtrip_rgb(rgb[0], streams=ref_zz, plan=plan)
        assert torch.equal(m.forward_rgb(rgb[0], streams=zz[0], plan=plan), ref_zz), "forward_rgb != fused streams"
        assert torch.equal(m.inverse_rgb(zz[0], out=out[0], plan=plan), ref), "inverse_rgb(forward_rgb) != roundtrip_rgb"
        del ref, ref_zz

        def pair(i):
            m.forward_rgb(rgb[i % 2], streams=zz[i % 2], plan=plan)
            m.inverse_rgb(zz[i % 2], out=out[i % 2], plan=plan)

        variants = (
            ("roundtrip_rgb", 6, lambda i: m.roundtrip_rgb(rgb[i % 2], out=out[i % 2], plan=plan)),
            ("roundtrip_rgb with streams", 12, lambda i: m.roundtrip_rgb(rgb[i % 2], out=out[i % 2], streams=zz[i % 2], plan=plan)),
            ("forward_rgb", 9, lambda i: m.forward_rgb(rgb[i % 2], streams=zz[i % 2], plan=plan)),
            ("inverse_rgb", 9, lambda i: m.inverse_rgb(zz[i % 2], out=out[i % 2], plan=plan)),
            ("forward_rgb + inverse_rgb", 18, pair),
        )
        lines.append(f"## {mode}")
        for name, bpp, fn in variants:
            us, lo, hi = time_window(fn, a.iters, a.reps, a.warmup)
            gbs = bpp * px / us / 1e3
            lines.append(f"{name:58s} {us:8.1f} us [{lo:.1f}, {hi:.1f}]  {bpp:2d} B/px {gbs:7.1f} GB/s  {gbs / COPY_PEAK_GBS:.3f} of the copy peak")
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
