#!/usr/bin/env python
"""The reference README's accuracy table (README.md:62-69: PEEN, MSE and compression factor for 6..10
retained coefficients and for the standard quantisation matrix), regenerated on the GPU.

    python benchmarks/readme_table.py [--size 2048] [--image file] [--colour] [--subsampling 420]

The README's "Circuit" image is not in the reference repository, so the default input is a
deterministic synthetic stand-in with the same character (dark background, straight traces and
pads with sharp edges, a soft illumination gradient, mild sensor noise) -- `circuit_like()` below.
Everything is computed by the library: fused round trip + MSE/PEEN inside the kernel
(b200dct_roundtrip_metrics), the zig-zag coefficient stream, and its baseline-JPEG coded size
(b200dct_zigzag_coded_bits);  CF = 8*H*W / coded bits.  "k coefficients" = the first k positions
of the zig-zag scan are kept (README.md:63), "Standard" = all 64."""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cuda_dct_idct_b200 as m  # noqa: E402


def circuit_like(n: int, seed: int = 7) -> np.ndarray:
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:n, 0:n].astype(np.float32)
    img = 40 + 25 * (xx / n) + 15 * np.sin(yy / n * 3.1)            # illumination
    for _ in range(n // 2):                                           # traces
        x0, y0 = rng.integers(0, n, 2)
        length, width = int(rng.integers(n // 32, n // 4)), int(rng.integers(2, 9))
        level = float(rng.integers(120, 230))
        if rng.random() < 0.5:
            img[y0:y0 + width, x0:x0 + length] = level
        else:
            img[y0:y0 + length, x0:x0 + width] = level
    for _ in range(n // 4):                                           # pads
        x0, y0, r = int(rng.integers(0, n)), int(rng.integers(0, n)), int(rng.integers(4, 12))
        img[(xx - x0) ** 2 + (yy - y0) ** 2 < r * r] = 245
    img += rng.normal(0, 4.0, img.shape)
    return img.clip(0, 255).astype(np.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=2048)
    ap.add_argument("--image", default=None, help="grayscale image file instead of the synthetic one")
    ap.add_argument("--colour", action="store_true", help="RGB version (three planes, chroma table)")
    ap.add_argument("--subsampling", choices=["444", "420"], default="444",
                    help="chroma of the RGB version: full resolution, or 4:2:0 as JPEG encoders do by default (implies --colour)")
    args = ap.parse_args()
    args.colour = args.colour or args.subsampling == "420"
    if args.image:
        img = m.imageio.load_gray(args.image)
        b = 16 if args.subsampling == "420" else 8
        img = np.ascontiguousarray(img[: img.shape[0] // b * b, : img.shape[1] // b * b])
    else:
        img = circuit_like(args.size)
    H, W = img.shape
    cols = [6, 7, 8, 9, 10, 64]
    rows = {"PEEN (%)": [], "MSE": [], "Compr. Factor": [], "non-zero coeff. / block": []}
    if not args.colour:
        d = torch.from_numpy(img).cuda()
        for k in cols:
            plan = m.Plan(keep=m.zigzag_mask(k), inverse=m.api.INVERSE_EXACT)
            zz = m.api.empty_zigzag(H, W, d.device)
            _, (mse, peen, nnz) = m.roundtrip_with_metrics(d, coef=zz, plan=plan, zigzag=True)
            rows["PEEN (%)"].append(peen)
            rows["MSE"].append(mse)
            rows["Compr. Factor"].append(m.compression_factor(zz))
            rows["non-zero coeff. / block"].append(nnz / (H * W / 64))
    else:
        rgb = np.stack([img, np.roll(img, 3, 0) // 2 + 60, 255 - np.roll(img, 5, 1)], -1).astype(np.uint8)
        d = torch.from_numpy(rgb).cuda()
        for k in cols:
            plan = m.Plan(keep=m.zigzag_mask(k), inverse=m.api.INVERSE_EXACT)
            if args.subsampling == "420":
                zz = m.forward_rgb420(d, plan=plan)
                out = m.inverse_rgb420(zz, plan=plan)
                nnz, blocks = sum(float((s != 0).sum().item()) for s in zz), 1.5 * H * W / 64
            else:
                zz = torch.empty(3, H // 8, W // 8, 64, dtype=torch.int16, device=d.device)
                out = m.roundtrip_rgb(d, streams=zz, plan=plan)
                nnz, blocks = float((zz != 0).sum().item()), 3 * H * W / 64
            mse, peen = m.metrics(d.view(H, W * 3), out.view(H, W * 3))
            rows["PEEN (%)"].append(peen)
            rows["MSE"].append(mse)
            rows["Compr. Factor"].append(m.compression_factor(zz))
            rows["non-zero coeff. / block"].append(nnz / blocks)
    kind = ("RGB 4:2:0" if args.subsampling == "420" else "RGB 4:4:4") if args.colour else "grayscale"
    print(f"Input: {'synthetic circuit-like' if not args.image else args.image} {H}x{W} {kind} u8; "
          "HpApprDCT (Haweel T), JPEG tables; CF = 8*H*W*channels / baseline-JPEG coded bits\n")
    print("| Metric / Coefficients | 6 | 7 | 8 | 9 | 10 | Standard |")
    print("| :--- | :---: | :---: | :---: | :---: | :---: | :---: |")
    for name, vals in rows.items():
        print(f"| **{name}** | " + " | ".join(f"{v:.2f}" for v in vals) + " |")


if __name__ == "__main__":
    main()
