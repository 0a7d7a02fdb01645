#!/usr/bin/env python
"""Writes tests/golden/libjpeg_420.npz: what the REAL libjpeg (libjpeg-turbo inside Pillow) computes when it
subsamples chroma 4:2:0 (h2v2), so the CPU suite can pin the 4:2:0 reference's two resamplers
(tests/rgb420_ref.py).  Both images are encoded at quality 100 (every Q entry 1) with subsampling=2 and decoded
with out_color_space = JCS_YCbCr (Pillow's draft("YCbCr")), i.e. after libjpeg's default upsampling.

  * down_rgb / down_swap_rgb : 16x16 MCUs built from 2x2 RGB groups whose full-resolution Cb samples sum to
    4k + 2 at even half-resolution columns and 4k + 1 at odd ones, and whose Cr samples sum to 4k' + 2 and
    4k' + 1 the same way.  With libjpeg's bias (1 at even columns, 2 at odd ones) every such group downsamples
    to k (k'): the half-resolution planes are constant, their blocks DC-only, which survives Q = 1 and the
    inverse DCT exactly.  down_ycc: the decoded planes.  down_swap_rgb has the same groups in swapped column
    order (down_swap_ycc its decode), which the bias turns into two values.
  * up_rgb : constant-colour 16x16 MCUs of random colours.  Every chroma block is DC-only, so the decoded
    half-resolution plane is exactly one sample per MCU (up_half, the Cb / Cr of that colour, as jccolor.c
    computes it), and up_ycc, the decoded full-resolution planes, is libjpeg's upsampling of it -- MCU
    boundaries and image edges included.
Run in the build container (needs Pillow); the output is committed."""
import io
import os

import numpy as np
from PIL import Image, features

HERE = os.path.dirname(os.path.abspath(__file__))


def ycc(rgb):
    """jccolor.c rgb_ycc_convert (16-bit fixed point), as the oracle restates it."""
    r, g, b = (rgb[..., c].astype(np.int64) for c in range(3))
    fix = lambda x: int(x * 65536 + 0.5)  # noqa: E731
    y = (fix(0.299) * r + fix(0.587) * g + fix(0.114) * b + 32768) >> 16
    cb = (-fix(0.16874) * r - fix(0.33126) * g + fix(0.5) * b + (128 << 16) + 32767) >> 16
    cr = (fix(0.5) * r - fix(0.41869) * g - fix(0.08131) * b + (128 << 16) + 32767) >> 16
    return np.stack([y, cb, cr], -1)


def decode_ycc(rgb):
    buf = io.BytesIO()
    Image.fromarray(rgb).save(buf, "JPEG", quality=100, subsampling=2)
    im = Image.open(io.BytesIO(buf.getvalue()))
    assert im.layer[0][1:3] == (2, 2) and im.layer[1][1:3] == (1, 1), "expected a 4:2:0 file"
    im.draft("YCbCr", im.size)
    assert im.mode == "YCbCr"
    return np.array(im)


def groups(rng, n):
    """n pairs of 2x2 RGB groups: (even, odd) with Cb sums 4k + 2 / 4k + 1 and Cr sums 4k' + 2 / 4k' + 1."""
    out = []
    while len(out) < n:
        base = rng.integers(40, 216, 3)
        cand = (base + rng.integers(-6, 7, (256, 4, 3))).astype(np.uint8)
        s = ycc(cand)[..., 1:].sum(1)                 # (256, 2): Cb, Cr sums of each candidate group
        even = np.flatnonzero(((s % 4) == 2).all(1))
        odd = np.flatnonzero(((s % 4) == 1).all(1))
        for e in even:
            match = odd[((s[odd] - 1) // 4 == (s[e] - 2) // 4).all(1)]
            if len(match):
                out.append((cand[e], cand[match[0]]))
                break
    return out


def main():
    rng = np.random.default_rng(420)
    # down: 6 x 10 MCUs, every MCU filled with one pair of groups (even, odd) tiled over its 8 x 8 chroma samples
    mh, mw = 6, 10
    pairs = groups(rng, mh * mw)
    down, swap = np.empty((mh * 16, mw * 16, 3), np.uint8), np.empty((mh * 16, mw * 16, 3), np.uint8)
    for i, (e, o) in enumerate(pairs):
        my, mx = divmod(i, mw)
        for img, (a, b) in ((down, (e, o)), (swap, (o, e))):
            tile = np.empty((2, 4, 3), np.uint8)      # one row pair of groups: columns 0-1 group a, 2-3 group b
            tile[:, 0:2] = a.reshape(2, 2, 3)
            tile[:, 2:4] = b.reshape(2, 2, 3)
            img[my * 16:(my + 1) * 16, mx * 16:(mx + 1) * 16] = np.tile(tile, (8, 4, 1))
    # up: 6 x 9 constant-colour MCUs, 96 x 144 pixels
    uh, uw = 6, 9
    cols = rng.integers(0, 256, (uh, uw, 3), dtype=np.uint8)
    up = np.repeat(np.repeat(cols, 16, 0), 16, 1)
    up_ycc = decode_ycc(up)
    half = ycc(cols)[..., 1:].astype(np.uint8)
    out = {"down_rgb": down, "down_ycc": decode_ycc(down), "down_swap_rgb": swap, "down_swap_ycc": decode_ycc(swap),
           "up_rgb": up, "up_half": half, "up_ycc": up_ycc,
           "libjpeg": np.array(f"{features.version('jpg')} turbo={features.check_feature('libjpeg_turbo')}")}
    np.savez_compressed(os.path.join(HERE, "libjpeg_420.npz"), **out)
    print({k: getattr(v, "shape", v) for k, v in out.items()})


if __name__ == "__main__":
    main()
