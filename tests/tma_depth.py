"""The persistent TMA kernels' tile loop at depth: shapes that put every warp through several tiles, the launch
geometry read back from a profiler trace, and the float64 bounds of tests/f64ref.py evaluated in bands.

k_tma (csrc/dct_kernels.cuh) runs one CTA per SM; its `grid x warps` warps draw 256-pixel-wide, 8-row tiles
from a ticket counter.  The first `grid x warps` tickets are pre-assigned, the counter hands out the rest: runs
of two tiles for the first `run_tickets` tickets, single tiles once no more than two rounds of the machine
remain (b200dct.cu run_tma).  With S = grid x warps and n tiles:
  R1  n <= S        every warp takes at most one tile: the loop body runs once (the small matrix cells);
  R2  S < n <= 2S   single tickets only: the barrier parity flips, buffers are reused, no run tickets;
  R3  n >= 3S + 1   run tickets, then a single-tile tail; with n - 2S odd the tail starts on an odd remainder.
The width of a deep shape is 32 (mod 256): its last tile column is a partial tile of four blocks.

Pure helpers (the shape arithmetic, the trace parser) import neither torch nor a device.
"""
from __future__ import annotations

import json
import os
import tempfile

import numpy as np

import f64ref as R

DEEP_W = 2080                    # 8 full tiles and a partial tile of 32 pixels per tile row
TILE_W = 256
BAND_ROWS = 1024                 # rows per band of the float64 checks (128 block rows)

# tile bytes of a plane element type, as in dct_core.cuh tile_bytes_of (8 rows x 256 pixels)
TILE_BYTES = {"f32": 8192, "i16": 4096, "u8": 2048}
SMEM_BYTES = 227 * 1024          # shared memory a CTA may opt into on a B200
METRICS_WARPS = 9                # TMA_METRICS_THREADS / 32


def tiles_x(W: int) -> int:
    return (W + TILE_W - 1) // TILE_W


def ntiles(H: int, W: int) -> int:
    return tiles_x(W) * (H // 8)


def cta_warps(pix: str, tk: int, planes: list[str], metrics: bool = False) -> int:
    """Warps per CTA of a k_tma launch: the flavour's CTA size (u8 pixels 16, Haweel's T 8, dense T 12, fused
    metrics 9), limited by the shared memory of (NIN + 1) tile buffers per warp, each as large as the largest tile
    of the call's planes.  The deep tests assert the resulting regime from the launch itself, so a mistake here
    shows up as a failed regime, never as a silently shallow test."""
    nw = METRICS_WARPS if metrics else (16 if pix == "u8" else 8 if tk == 1 else 12)
    buf = max(TILE_BYTES[p] for p in planes)
    nbuf = 3 if metrics else 2
    return min(nw, (SMEM_BYTES - 1024) // (nbuf * buf + 16))


def deep_height(sms: int, warps: int, W: int = DEEP_W) -> int:
    """The smallest H (a multiple of 8) with n >= 3S + 1 and n - 2S odd, S = sms x warps (regime R3)."""
    tx, S = tiles_x(W), sms * warps
    hb = -(-(3 * S + 1) // tx)
    while (tx * hb - 2 * S) % 2 == 0:
        hb += 1
    return 8 * hb


def r2_height(sms: int, warps: int, W: int = DEEP_W) -> int:
    """An H with S < n <= 2S (regime R2), n near 1.5 S."""
    tx, S = tiles_x(W), sms * warps
    hb = max(1, (3 * S // 2) // tx)
    assert S < tx * hb <= 2 * S, (sms, warps, W)
    return 8 * hb


def regime(n: int, grid: int, block: int) -> str:
    S = grid * (block // 32)
    if n <= S:
        return "R1"
    if n <= 2 * S:
        return "R2"
    return "R3" if n >= 3 * S + 1 and (n - 2 * S) % 2 == 1 else "between"


# ---------------------------------------------------------------- launch geometry from the profiler
def kernel_geometry(trace: dict) -> list[tuple[str, tuple, tuple]]:
    """(name, grid, block) of every kernel event of a chrome trace exported by torch.profiler.  A kernel event
    without `grid` or `block` raises: the regime of a deep test cannot be proved without them."""
    out = []
    for ev in trace.get("traceEvents", []):
        if ev.get("cat") != "kernel":
            continue
        args = ev.get("args", {})
        if "grid" not in args or "block" not in args:
            raise AssertionError(f"the profiler trace carries no grid / block for kernel {ev.get('name')!r}: "
                                 f"args {sorted(args)}")
        out.append((ev["name"], tuple(args["grid"]), tuple(args["block"])))
    return out


def warm_up():
    """One small torch kernel at the start of a profiler session, completed before the kernels under test run.
    CUPTI sometimes asks for a new activity buffer at a session's first kernel and that kernel's record is lost
    (the session then shows an 'Activity Buffer Request' and no kernel); the warm-up kernel takes that place."""
    import torch

    torch.ones(1, device="cuda").add_(1)
    torch.cuda.synchronize()


def profiled(fn):
    """fn() under torch.profiler (CUDA activity only): (fn's result, the profile, [(name, grid, block)])."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        warm_up()
        res = fn()
        torch.cuda.synchronize()
    fd, path = tempfile.mkstemp(suffix=".json")
    os.close(fd)
    try:
        prof.export_chrome_trace(path)
        with open(path) as f:
            geo = kernel_geometry(json.load(f))
    finally:
        os.unlink(path)
    return res, prof, geo


def tma_launch(geo, canonical) -> tuple[str, int, int]:
    """(key, grid, block) of the one k_tma launch among the profiled kernels."""
    tma = [(canonical(n), g, b) for n, g, b in geo if canonical(n).startswith("k_tma<")]
    assert len(tma) == 1, f"expected one k_tma launch, got {[t[0] for t in tma]}"
    key, g, b = tma[0]
    assert g[1:] == (1, 1) and b[1:] == (1, 1), f"{key}: grid {g}, block {b}"
    return key, g[0], b[0]


# ---------------------------------------------------------------- float64 bounds in bands of block rows
def _bands(H: int, rows: int = BAND_ROWS):
    for r0 in range(0, H, rows):
        yield slice(r0, min(H, r0 + rows))


def _merge(parts: list[R.Check]) -> R.Check:
    n = sum(p.n for p in parts)
    amb = sum(p.ambiguous * p.n for p in parts) / max(1, n)
    return R.Check(sum(p.bad for p in parts), amb, max((p.worst for p in parts), default=0.0), n)


def check_quant_banded(coef, img, T, Q, keep) -> R.Check:
    """f64ref.check_quant of a whole coefficient plane against forward64 of the whole image, a band at a time."""
    parts = []
    for b in _bands(img.shape[0]):
        Y, B = R.forward64(img[b], T)
        parts.append(R.check_quant(coef[b], Y, B, Q, keep))
    return _merge(parts)


def check_pixels_banded(got, C, T, Q) -> R.Check:
    """Pixels of a re-associated inverse (f32: check_close, u8: check_u8) against inverse64 of the coefficients
    C, a band at a time."""
    parts = []
    for b in _bands(got.shape[0]):
        P, Bi = R.inverse64(C[b], T, Q)
        parts.append(R.check_u8(got[b], P, Bi) if got.dtype == np.uint8 else R.check_close(got[b], P, Bi))
    return _merge(parts)
