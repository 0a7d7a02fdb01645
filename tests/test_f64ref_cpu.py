"""CPU: the float64 reference and error bounds of tests/f64ref.py.

The bit-exact chain oracle and numpy f32 emulations of the re-associated kernels (written line by line
from dct_core.cuh and mma_kernels.cuh) must pass every checker; deliberately wrong variants of them
must fail at least one.  That shows the bounds hold for the arithmetic the kernels run and that the
checkers have teeth.  An fma is emulated as the float64 product-sum rounded once to f32."""
from __future__ import annotations

import numpy as np
import pytest

import f64ref as R
import inputs

F32 = np.float32
SCALES = [-12, -6, -1, 0, 3, 8, 12, 16]     # as tests/test_gpu_range.py: x_s = 128 + 2^k (x0 - 128), Q_s = 2^k Q
MAX_AMBIGUOUS = 1e-2
MAX_AMBIGUOUS_MMA = 5e-2    # the bound is 4.5 times wider, and so is the band around each half-integer


def fma(a, b, c):
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(F32)


def f32(v):
    return np.float32(v)


# ---------------------------------------------------------------- emulations of the kernels
def quantise(y, Q, keep=R.ALL_COEFFS, half_even=False):
    """quantise() of dct_core.cuh on (nb, 8, 8) blocks: correctly rounded y/Q, round half away."""
    q = (y.astype(np.float64) / R.q_grid(Q)).astype(F32).astype(np.float64)
    c = np.round(q) if half_even else R.round_half_away(q)
    return np.where(R.keep_grid(keep), c, 0.0).astype(F32)


def forward_sym(x, T, Q, keep=R.ALL_COEFFS, half_even=False, Tq=None):
    """forward_block_sym: x = pixels - 128 as (nb, 8, 8) f32."""
    t = np.asarray(T, F32).reshape(8, 8)
    M = np.empty_like(x)
    sd = [x[:, n, :] + x[:, 7 - n, :] for n in range(4)] + [x[:, n, :] - x[:, 7 - n, :] for n in range(4)]
    for k in range(8):
        base = (k & 1) * 4
        acc = sd[base] * t[k, 0]
        for n in range(3):
            acc = fma(sd[base + 1 + n], t[k, 1 + n], acc)
        M[:, k, :] = acc
    Y = np.empty_like(x)
    # row pass: {s_n, d_n} = fma(r[7-n], {1, -1}, r[n]); {y[2i], y[2i+1]} from the (even, odd) pair eo
    s = [fma(M[:, :, 7 - n], 1.0, M[:, :, n]) for n in range(4)]
    d = [fma(M[:, :, 7 - n], -1.0, M[:, :, n]) for n in range(4)]
    for i in range(4):
        ax, ay = s[0] * t[2 * i, 0], d[0] * t[2 * i + 1, 0]
        for n in range(3):
            ax = fma(s[1 + n], t[2 * i, 1 + n], ax)
            ay = fma(d[1 + n], t[2 * i + 1, 1 + n], ay)
        Y[:, :, 2 * i], Y[:, :, 2 * i + 1] = ax, ay
    return quantise(Y, Q if Tq is None else Tq, keep, half_even)


def inverse_sym(C, T, Q):
    """inverse_block_sym: quantised (nb, 8, 8) -> pixels, +128 included."""
    t = np.asarray(T, F32).reshape(8, 8)
    D = (C * np.asarray(Q, F32).reshape(8, 8)).astype(F32)
    M = np.empty_like(D)
    for n in range(4):
        e, o = D[:, 0, :] * t[0, n], D[:, 1, :] * t[1, n]
        for i in range(3):
            e = fma(D[:, 2 + 2 * i, :], t[2 + 2 * i, n], e)
            o = fma(D[:, 3 + 2 * i, :], t[3 + 2 * i, n], o)
        M[:, n, :], M[:, 7 - n, :] = e + o, e - o
    X = np.empty_like(D)
    for n in range(4):
        ex, ey = fma(M[:, :, 0], t[0, n], 128.0), fma(M[:, :, 1], t[1, n], 0.0)
        for i in range(3):
            ex = fma(M[:, :, 2 + 2 * i], t[2 + 2 * i, n], ex)
            ey = fma(M[:, :, 3 + 2 * i], t[3 + 2 * i, n], ey)
        X[:, :, n], X[:, :, 7 - n] = ex + ey, ex - ey
    return X


HA, HH, HP, HQ, HS = f32(0.35355339), f32(0.5), f32(0.4472136), f32(0.2236068), f32(0.70710678)


def inverse_fast(C, Q, bias_twice=False):
    """inverse_block_fast<true>: Haweel's T, quantised (nb, 8, 8) -> pixels, +128 on the DC term."""
    D = (C * np.asarray(Q, F32).reshape(8, 8)).astype(F32)
    c = [D[:, k, :] for k in range(8)]
    u = c[0] * HA
    A, B = fma(c[4], HA, u), fma(c[4], -HA, u)
    P, Rr = fma(c[6], HQ, c[2] * HP), fma(c[6], -HP, c[2] * HQ)
    E0, E3, E1, E2 = A + P, A - P, B + Rr, B - Rr
    sm, df = c[1] + c[5], c[1] - c[5]
    M = np.empty_like(D)
    M[:, 0, :], M[:, 7, :] = fma(sm, HH, E0), fma(sm, -HH, E0)
    M[:, 1, :], M[:, 6, :] = fma(df, HH, E1), fma(df, -HH, E1)
    M[:, 2, :], M[:, 5, :] = fma(c[3], -HS, E2), fma(c[3], HS, E2)
    M[:, 3, :], M[:, 4, :] = fma(c[7], -HS, E3), fma(c[7], HS, E3)
    m = [M[:, :, k] for k in range(8)]
    u = fma(m[0], HA, 128.0)
    A, B = fma(m[4], HA, u), fma(m[4], -HA, u)                       # AB = ffma2(m4, {a,-a}, u)
    if bias_twice:
        A = (A + f32(128.0)).astype(F32)
    P, Rr = fma(m[6], HQ, m[2] * HP), fma(m[6], -HP, m[2] * HQ)      # PR
    s_, d_ = fma(m[5], 1.0, m[1]), fma(m[5], -1.0, m[1])             # SD
    E0, E3 = fma(P, 1.0, A), fma(P, -1.0, A)
    E1, E2 = fma(Rr, 1.0, B), fma(Rr, -1.0, B)
    X = np.empty_like(D)
    X[:, :, 0], X[:, :, 7] = fma(s_, HH, E0), fma(s_, -HH, E0)
    X[:, :, 1], X[:, :, 6] = fma(d_, HH, E1), fma(d_, -HH, E1)
    X[:, :, 2], X[:, :, 5] = fma(-m[3], HS, E2), fma(-m[3], -HS, E2)
    X[:, :, 3], X[:, :, 4] = fma(-m[7], HS, E3), fma(-m[7], -HS, E3)
    return X


def tf32_rna(v):
    b = np.asarray(v, F32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(F32)


def tf32_trunc(v):
    return (np.asarray(v, F32).view(np.uint32) & np.uint32(0xFFFFE000)).view(F32)


def mma_pass(L, V, lo=True):
    """mma_pass: L . V for (nb, 8, 8) V.  A = [L_hi ; L_lo]; V issued as v_hi and v - v_hi (the MMA
    reads its TF32 bits); each MMA accumulates its 8 products onto d with one rounding (one of the
    orders the bound allows); rows m and m+8 added in f32."""
    L = np.asarray(L, F32)
    lh = tf32_rna(L)
    ll = tf32_rna((L - lh).astype(F32))
    vh = tf32_rna(V)
    vl = tf32_trunc((V - vh).astype(F32))
    d_hi = (lh.astype(np.float64) @ vh.astype(np.float64)).astype(F32)
    if not lo:
        return d_hi
    d_hi = (d_hi + lh.astype(np.float64) @ vl.astype(np.float64)).astype(F32)
    d_lo = (ll.astype(np.float64) @ vh.astype(np.float64)).astype(F32)
    d_lo = (d_lo + ll.astype(np.float64) @ vl.astype(np.float64)).astype(F32)
    return (d_hi + d_lo).astype(F32)


def mma_roundtrip(x, T, Q, keep=R.ALL_COEFFS, lo=True):
    """k_mma on (nb, 8, 8) pixels-128: returns (coefficients, pixels)."""
    t = np.asarray(T, F32).reshape(8, 8)
    M = mma_pass(t, x, lo)
    Y = mma_pass(t, M.transpose(0, 2, 1), lo).transpose(0, 2, 1)
    C = quantise(Y, Q, keep)
    D = (C * np.asarray(Q, F32).reshape(8, 8)).astype(F32)
    M2 = mma_pass(t.T, D, lo)
    Rt = mma_pass(t.T, M2.transpose(0, 2, 1), lo).transpose(0, 2, 1)
    return C, (Rt + f32(128.0)).astype(F32)


# ---------------------------------------------------------------- inputs
def standard_images(oracle):
    return {
        "rand": oracle.rand_image(128, 256, 42),
        "adversarial": inputs.adversarial(32),
        "float_noise": inputs.float_noise(128, 256),
        "smooth": inputs.smooth_image(128, 256),
    }


def all_images(oracle):
    imgs = standard_images(oracle)
    rng = np.random.default_rng(4)
    imgs["pm1e4"] = (rng.random((64, 256)) * 2e4 - 1e4).astype(F32)
    x0 = rng.integers(0, 256, (256, 256)).astype(F32)
    x0[:128] = inputs.adversarial(32)
    for k in SCALES:
        s = F32(2.0 ** k)
        imgs[f"scale{k}"] = (F32(128) + s * (x0 - F32(128))).astype(F32)
    return imgs


def q_for(name, oracle):
    k = int(name[5:]) if name.startswith("scale") else 0
    return (oracle.jpeg_Q() * F32(2.0 ** k)).astype(F32)


def unquantised(oracle, img, T, B):
    """The oracle's f32 Y: Q = 2^-k with Y 2^k < 2^100 makes the quantised value round(Y 2^k), which is
    Y 2^k itself down to 2^-(k+1) absolute (far below u B wherever B > 0)."""
    k = 100 - int(np.ceil(np.log2(max(float(B.max()), 1e-30))))
    return oracle.dct(img, T=T, Q=np.full(64, 2.0 ** -k, F32)).astype(np.float64) * 2.0 ** -k


# ---------------------------------------------------------------- 1. the oracle passes
@pytest.mark.parametrize("tname", ["haweel", "dct2"])
def test_chain_oracle_passes_every_checker(oracle, tname):
    T = oracle.haweel_T() if tname == "haweel" else oracle.dct2_T()
    worst = {"Y": 0.0, "f32": 0.0, "amb": 0.0}
    for name, img in all_images(oracle).items():
        Q = q_for(name, oracle)
        Y, B = R.forward64(img, T)
        fy = R.check_close(unquantised(oracle, img, T, B), Y, B, R.C_F)
        assert fy.bad == 0, (name, str(fy))
        coef = oracle.dct(img, T=T, Q=Q)
        cq = R.check_quant(coef, Y, B, Q)
        assert cq.bad == 0, (name, str(cq))
        assert cq.ambiguous <= MAX_AMBIGUOUS, (name, str(cq))
        P, Bi = R.inverse64(coef, T, Q)
        pix = oracle.idct(coef, T=T, Q=Q)
        cp = R.check_close(pix, P, Bi)
        assert cp.bad == 0, (name, str(cp))
        cu = R.check_u8(oracle.to_u8(pix), P, Bi)
        assert cu.bad == 0, (name, str(cu))
        worst = {"Y": max(worst["Y"], fy.worst), "f32": max(worst["f32"], cp.worst), "amb": max(worst["amb"], cq.ambiguous)}
    print(f"[f64ref] oracle {tname}: forward {worst['Y']:.2f} uB, inverse {worst['f32']:.2f} uB, ambiguous <= {worst['amb']:.2e}")
    assert worst["Y"] > 0 and worst["f32"] > 0      # the checks see the f32 rounding at all


def test_oracle_reaches_the_bound_far_from_its_limit(oracle):
    """The derivation gives ~19 u B for the chains; the oracle stays well inside (a bound that the
    reference itself nearly hits would leave no room for the re-associated kernels)."""
    T = oracle.haweel_T()
    img = oracle.rand_image(256, 256, 3)
    Y, B = R.forward64(img, T)
    assert R.check_close(unquantised(oracle, img, T, B), Y, B, R.C_F / 4).bad == 0


# ---------------------------------------------------------------- 2. emulations pass
def _blocks(img):
    return R.to_blocks((img - F32(128)).astype(F32))


@pytest.mark.parametrize("tname", ["dct2", "randsym"])
def test_symmetric_emulation_passes(oracle, tname):
    T = oracle.dct2_T() if tname == "dct2" else R.rand_sym_T()
    for name, img in all_images(oracle).items():
        Q = q_for(name, oracle)
        H, W = img.shape
        Y, B = R.forward64(img, T)
        C = R.from_blocks(forward_sym(_blocks(img), T, Q), H, W)
        cq = R.check_quant(C, Y, B, Q)
        assert cq.bad == 0 and cq.ambiguous <= MAX_AMBIGUOUS, (name, str(cq))
        P, Bi = R.inverse64(C, T, Q)
        pix = R.from_blocks(inverse_sym(R.to_blocks(C), T, Q), H, W)
        assert R.check_close(pix, P, Bi).bad == 0, name
        assert R.check_u8(oracle.to_u8(pix), P, Bi).bad == 0, name


def test_factored_inverse_emulation_passes(oracle):
    T = oracle.haweel_T()
    for name, img in all_images(oracle).items():
        Q = q_for(name, oracle)
        H, W = img.shape
        coef = oracle.dct(img, T=T, Q=Q)
        P, Bi = R.inverse64(coef, T, Q)
        pix = R.from_blocks(inverse_fast(R.to_blocks(coef), Q), H, W)
        cp = R.check_close(pix, P, Bi)
        assert cp.bad == 0, (name, str(cp))
        assert R.check_u8(oracle.to_u8(pix), P, Bi).bad == 0, name


def test_mma_emulation_passes(oracle):
    T = oracle.dct2_T()
    for name, img in all_images(oracle).items():
        Q = q_for(name, oracle)
        H, W = img.shape
        Y, B = R.forward64(img, T)
        C, pix = mma_roundtrip(_blocks(img), T, Q)
        C, pix = R.from_blocks(C, H, W), R.from_blocks(pix, H, W)
        cq = R.check_quant(C, Y, B, Q, c=R.C_MMA)
        assert cq.bad == 0 and cq.ambiguous <= MAX_AMBIGUOUS_MMA, (name, str(cq))
        P, Bi = R.inverse64(C, T, Q)
        cp = R.check_close(pix, P, Bi, R.C_MMA)
        assert cp.bad == 0, (name, str(cp))


def test_check_helpers(oracle):
    assert np.array_equal(R.round_half_away(np.array([-2.5, -0.5, 0.5, 1.5, 2.49])), [-3, -1, 1, 2, 2])
    img = oracle.rand_image(16, 24, 1)
    coef = oracle.dct(img)
    assert np.array_equal(R.unzigzag(oracle.zigzag_i16(coef)), coef)
    # u8: a value a hair below an integer is admissible either side, one clearly inside is not
    P = np.array([[99.9999999, 99.5, 256.0, -3.0]])
    want, amb, other = R.expected_u8(P, np.full_like(P, 1000.0))
    assert want.tolist() == [[99, 99, 255, 0]] and amb.tolist() == [[True, False, False, False]] and other[0, 0] == 100
    # f32: a NaN (an output left at its sentinel) or an infinity is outside every bound, however wide
    exact = np.array([1.0, 2.0, 3.0, 4.0])
    got = np.array([1.0, np.nan, np.inf, 4.0], np.float32)
    assert R.check_close(got, exact, np.full(4, 1e30)).bad == 2
    assert R.check_close(exact.astype(np.float32), exact, np.ones(4)).bad == 0


# ---------------------------------------------------------------- 3. mutants fail
def _rejected(checks):
    return any(c.bad > 0 for c in checks)


def _sym_checks(oracle, T_true, T_used, Q, Q_used=None, half_even=False):
    out = []
    for img in standard_images(oracle).values():
        H, W = img.shape
        Y, B = R.forward64(img, T_true)
        C = R.from_blocks(forward_sym(_blocks(img), T_used, Q, half_even=half_even, Tq=Q_used), H, W)
        out.append(R.check_quant(C, Y, B, Q))
        P, Bi = R.inverse64(C, T_true, Q)
        pix = R.from_blocks(inverse_sym(R.to_blocks(C), T_used, Q), H, W)
        out += [R.check_close(pix, P, Bi), R.check_u8(oracle.to_u8(pix), P, Bi)]
    return out


def test_mutant_T_constant_off_by_2_pow_minus_12(oracle):
    T = oracle.dct2_T()
    assert not _rejected(_sym_checks(oracle, T, T, oracle.jpeg_Q()))
    bad = T.copy()
    bad[2 * 8 + 1] *= F32(1 + 2.0 ** -12)
    bad[2 * 8 + 6] = bad[2 * 8 + 1]              # keeps the symmetry, so the same kernel would run
    assert _rejected(_sym_checks(oracle, T, bad, oracle.jpeg_Q()))


def test_mutant_transposed_Q(oracle):
    T, Q = oracle.dct2_T(), oracle.jpeg_Q()
    assert _rejected(_sym_checks(oracle, T, T, Q, Q_used=Q.reshape(8, 8).T.reshape(64)))


def test_mutant_round_half_even(oracle):
    """A tie is only decidable where the arithmetic is exact: any sound bound admits both neighbours of
    a tie that f32 rounding may have produced.  With T in multiples of 1/8 (the DCT-II rounded, so the
    symmetric kernels apply) and integer pixels every sum is exact in f32 (|Y| < 2^13 in steps of
    2^-6), so the checker may run with c = 0: then the exact ties of the adversarial and random bands
    must round away from zero."""
    T = (np.round(oracle.dct2_T() * 8) / 8).astype(F32)
    Q = oracle.jpeg_Q()
    img = np.concatenate([inputs.adversarial(32), oracle.rand_image(64, 256, 42)])
    Y, B = R.forward64(img, T)
    z = Y / R.tile(R.q_grid(Q), *img.shape)
    assert np.count_nonzero(np.abs(z - np.floor(z)) == 0.5) > 0       # exact ties exist
    H, W = img.shape
    good = R.from_blocks(forward_sym(_blocks(img), T, Q), H, W)
    assert R.check_quant(good, Y, B, Q, c=0).bad == 0
    even = R.from_blocks(forward_sym(_blocks(img), T, Q, half_even=True), H, W)
    assert R.check_quant(even, Y, B, Q, c=0).bad > 0
    assert R.check_quant(even, Y, B, Q).bad == 0      # with the general bound a tie admits both answers


def test_mutant_mma_without_lo_terms(oracle):
    T = oracle.dct2_T()
    checks = []
    for img in standard_images(oracle).values():
        H, W = img.shape
        Y, B = R.forward64(img, T)
        C, pix = mma_roundtrip(_blocks(img), T, oracle.jpeg_Q(), lo=False)
        C, pix = R.from_blocks(C, H, W), R.from_blocks(pix, H, W)
        P, Bi = R.inverse64(C, T, oracle.jpeg_Q())
        checks += [R.check_quant(C, Y, B, oracle.jpeg_Q(), c=R.C_MMA), R.check_close(pix, P, Bi, R.C_MMA)]
    assert _rejected(checks)


def test_mutant_factored_inverse_with_double_bias(oracle):
    T, Q = oracle.haweel_T(), oracle.jpeg_Q()
    checks = []
    for img in standard_images(oracle).values():
        H, W = img.shape
        coef = oracle.dct(img, T=T, Q=Q)
        P, Bi = R.inverse64(coef, T, Q)
        pix = R.from_blocks(inverse_fast(R.to_blocks(coef), Q, bias_twice=True), H, W)
        checks += [R.check_close(pix, P, Bi), R.check_u8(oracle.to_u8(pix), P, Bi)]
    assert _rejected(checks)
