"""Float64 reference of the 8x8 block transform and a-priori error bounds for the kernels that
re-associate their f32 sums (numpy only).

The exact-chain kernels are pinned bit for bit to the CPU oracle.  Four arithmetics are not: the
even/odd evaluation of a symmetric dense T (dct_core.cuh forward_block_sym / inverse_block_sym), the
factored inverse of Haweel's T (inverse_block_fast), the tensor-core arm (mma_kernels.cuh) and the
colour inverse that uses the factored inverse.  Their contract is a bound against EXACT arithmetic:

    |computed - exact| <= c * u * B,   u = 2^-24 (unit roundoff of f32, round to nearest)

with B the same sum taken over absolute values.  The checkers below compare with a float64
evaluation of the plan's own f32 T and Q (float64 holds every product of two f32 exactly, and its own
rounding, ~2^-53 relative, is far below u).  There is no statistical allowance: any value outside the
bound fails, wherever it is.

Derivation of the constants (first order in u; the u^2 terms are < 1e-5 of the bound).

CUDA-core kernels.  An inner product evaluated by k dependent roundings of which each term passes
through at most k has |err| <= gamma_k * sum|a_i b_i|, gamma_k = k u / (1 - k u)  (Higham, "Accuracy and
Stability of Numerical Algorithms", 3.1).  Depth per pass, counted from dct_core.cuh:
  * ordered chain: 8 FMAs;
  * forward_block_sym: one pre-add (x[n] +- x[7-n]) then a 4-term FMA chain: 5;
  * inverse_block_sym: a 4-term chain then the final E +- O add: 5;
  * inverse_block_fast: the deepest term (c2: mul, fma, add, fma) is rounded 4 times.
So 9 covers every pass.  Forward: X - 128 in f32 (one rounding, u |X-128|; exact for u8 and
integer pixels), two passes: |Y_f32 - Y| <= (u + 2 gamma_9 + gamma_9^2) B  ~ 19.0 u B.  The quantiser
divides correctly rounded (u |z|) and rounds half away from zero exactly, so with z = Y/Q
    |z_f32 - z| <= 19 u B / |Q| + u (|z| + 19 u B/|Q|)  <=  C_F u B/|Q| + 2 u |z|,   C_F = 20.
Where no half-integer lies within that distance of z, the quantised value is round_half_away(z).
Inverse: C*Q (u |C Q|), two passes (2 gamma_9), the +128 (folded into a chain, or one add: u |R+128|):
    |P_f32 - P| <= 20 u Bi,  Bi = |T|^T |C Q| |T| + 128,   C_I = 20.

Tensor-core arm (k_mma, mma_kernels.cuh:16-20).  One pass L.v on m16n8k8 TF32 MMAs with
A = [L_hi ; L_lo] and v issued as v_hi then v - v_hi:
  * L_hi = rna_tf32(L), L_lo = rna_tf32(L - L_hi): |L - L_hi - L_lo| <= 2^-11 |L - L_hi| <= 2^-22 |L| = 4 u |L|;
  * v_hi = rna_tf32(v): |v - v_hi| <= 2^-11 |v|; the MMA reads only the TF32 bits of v - v_hi, i.e. it
    TRUNCATES it to 10 mantissa bits: lost <= 2^-10 |v - v_hi| <= 2^-21 |v| = 8 u |v|;
  * products of two TF32 values are exact in FP32; the accumulation order and rounding inside the tensor
    core are not specified: allow any order and round-toward-zero (2u per addition).  16 products per
    output (two MMAs of k = 8) need at most 15 additions on any path: 30 u;
  * rows m and m+8 added on the CUDA cores: u.
Per pass 4 + 8 + 30 + 1 = 43 u of |L| |v|.  Forward: X - 128 (u) and two passes: 87 u B, plus the
quantiser as above.  Inverse: C*Q (u), two passes, +128 (u): 88 u Bi.  C_MMA = 90 covers both.

No constant here is fitted to GPU output.
"""
from __future__ import annotations

from typing import NamedTuple

import numpy as np

U = 2.0 ** -24
C_F = 20.0
C_I = 20.0
C_MMA = 90.0
ALL_COEFFS = (1 << 64) - 1


def rand_sym_T(seed: int = 5) -> np.ndarray:
    """A T with the DCT-II symmetry (even rows symmetric, odd rows antisymmetric) whose row 0 is not
    constant, so that the +128 of inverse_block_sym meets a DC basis function unlike the DCT-II's."""
    rng = np.random.default_rng(seed)
    h = rng.uniform(-0.6, 0.6, (8, 4)).astype(np.float32)
    t = np.concatenate([h, h[:, ::-1]], 1)
    t[1::2, 4:] *= -1
    return t.reshape(64).astype(np.float32)


# ---------------------------------------------------------------- block layout
def to_blocks(a: np.ndarray) -> np.ndarray:
    """(H, W) -> (H/8 * W/8, 8, 8), blocks in raster order."""
    H, W = a.shape
    return a.reshape(H // 8, 8, W // 8, 8).transpose(0, 2, 1, 3).reshape(-1, 8, 8)


def from_blocks(b: np.ndarray, H: int, W: int) -> np.ndarray:
    return b.reshape(H // 8, W // 8, 8, 8).transpose(0, 2, 1, 3).reshape(H, W)


def _t64(T) -> np.ndarray:
    return np.asarray(T, np.float32).reshape(8, 8).astype(np.float64)


def q_grid(Q) -> np.ndarray:
    return np.asarray(Q, np.float32).reshape(8, 8).astype(np.float64)


def keep_grid(keep: int) -> np.ndarray:
    return np.array([(keep >> k) & 1 for k in range(64)], bool).reshape(8, 8)


# ---------------------------------------------------------------- the reference
def forward64(img: np.ndarray, T):
    """Y = T (X - 128) T^T per 8x8 block and B = |T| |X - 128| |T|^T, float64, (H, W) each.
    `img`: f32 or u8 pixels as the kernel reads them."""
    H, W = img.shape
    t = _t64(T)
    x = to_blocks(img.astype(np.float64) - 128.0)
    Y = t @ x @ t.T
    B = np.abs(t) @ np.abs(x) @ np.abs(t).T
    return from_blocks(Y, H, W), from_blocks(B, H, W)


def inverse64(C: np.ndarray, T, Q):
    """P = T^T (C o Q) T + 128 per block and Bi = |T|^T |C o Q| |T| + 128, float64, (H, W) each.
    `C`: a quantised coefficient plane (H, W)."""
    H, W = C.shape
    t = _t64(T)
    d = to_blocks(C.astype(np.float64)) * q_grid(Q)
    P = t.T @ d @ t + 128.0
    Bi = np.abs(t).T @ np.abs(d) @ np.abs(t) + 128.0
    return from_blocks(P, H, W), from_blocks(Bi, H, W)


def round_half_away(z: np.ndarray) -> np.ndarray:
    return np.sign(z) * np.floor(np.abs(z) + 0.5)


def tile(g: np.ndarray, H: int, W: int) -> np.ndarray:
    """An (8, 8) per-position table repeated over an (H, W) plane."""
    return np.tile(g, (H // 8, W // 8))


# ---------------------------------------------------------------- checkers
class Check(NamedTuple):
    bad: int          # positions outside the bound (must be 0)
    ambiguous: float  # fraction of positions where the bound admits two answers
    worst: float      # largest observed error in units of u * B (u8 / quantiser: implied by a flip; 0 if none)
    n: int

    def __str__(self):
        return f"bad={self.bad}/{self.n} ambiguous={self.ambiguous:.2e} worst={self.worst:.2f} uB"


def check_quant(coef: np.ndarray, Y: np.ndarray, B: np.ndarray, Q, keep: int = ALL_COEFFS, c: float = C_F) -> Check:
    """Quantised coefficients of a kernel against the exact Y (forward64).  Outside the keep mask they
    must be exactly 0.  Inside, with z = Y/Q and e = c u B/|Q| + 2 u |z|: where no half-integer lies
    within e of z the value must be round_half_away(z), elsewhere floor(z) or ceil(z).
    c = 0 declares the sums exact (tests that prove it); then only the correctly rounded division is
    left, which is exact wherever z is an f32 value."""
    H, W = coef.shape
    q = tile(q_grid(Q), H, W)
    kp = tile(keep_grid(keep), H, W)
    z = Y / q
    e = c * U * B / np.abs(q) + 2 * U * np.abs(z)
    if c == 0:
        e = np.where(z.astype(np.float32).astype(np.float64) == z, 0.0, e)
    got = coef.astype(np.float64)
    want = round_half_away(z)
    dist = np.abs(np.abs(z - np.floor(z)) - 0.5)            # distance to the nearest half-integer
    amb = (dist <= e) & (e > 0) & kp
    ok_amb = (got == np.floor(z)) | (got == np.ceil(z))
    ok = np.where(kp, (got == want) | (amb & ok_amb), got == 0)
    flips = kp & (got != want) & ok
    worst = float(np.max(dist[flips] * np.abs(q[flips]) / (U * B[flips]))) if flips.any() else 0.0
    return Check(int((~ok).sum()), float(amb.sum()) / max(1, int(kp.sum())), worst, coef.size)


def check_close(got: np.ndarray, exact: np.ndarray, mag: np.ndarray, c: float = C_I) -> Check:
    """f32 values (pixels from inverse64, or unquantised Y from forward64) within c u mag of exact."""
    err = np.abs(got.astype(np.float64) - exact)
    ratio = err / (U * np.maximum(mag, np.finfo(np.float64).tiny))
    return Check(int((err > c * U * mag).sum()), 0.0, float(ratio.max()) if ratio.size else 0.0, got.size)


def expected_u8(P: np.ndarray, Bi: np.ndarray, c: float = C_I):
    """(expected u8, ambiguous mask, the other admissible value) for exact pixels P: the library
    stores u8 as clamp to [0, 255] then truncate; where an integer k in [1, 255] lies within c u Bi of
    P either k - 1 or k is admissible."""
    want = np.trunc(np.clip(P, 0.0, 255.0))
    k = np.clip(np.rint(P), 1.0, 255.0)
    amb = np.abs(P - k) <= c * U * Bi
    other = np.where(want == k, k - 1, k)
    return want.astype(np.uint8), amb, np.where(amb, other, want).astype(np.uint8)


def check_u8(got: np.ndarray, P: np.ndarray, Bi: np.ndarray, c: float = C_I) -> Check:
    want, amb, other = expected_u8(P, Bi, c)
    ok = (got == want) | (amb & (got == other))
    flips = ok & (got != want)
    k = np.clip(np.rint(P), 1.0, 255.0)
    worst = float(np.max(np.abs(P - k)[flips] / (U * Bi[flips]))) if flips.any() else 0.0
    return Check(int((~ok).sum()), float(amb.mean()), worst, got.size)


# ---------------------------------------------------------------- zig-zag streams
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5,
                   12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
                   35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                   58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63])


def unzigzag(stream: np.ndarray) -> np.ndarray:
    """(H/8, W/8, 64) int16 zig-zag stream -> (H, W) float32 coefficient plane."""
    hb, wb, _ = stream.shape
    blk = np.zeros((hb, wb, 64), np.float32)
    blk[:, :, ZIGZAG] = stream
    return blk.reshape(hb, wb, 8, 8).transpose(0, 2, 1, 3).reshape(hb * 8, wb * 8)
