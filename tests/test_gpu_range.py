"""The f32 and int16 paths beyond the 8-bit range: pixels from 2^-10 to 2^23 with the quantiser scaled
alike, negative quantisers, coefficients that saturate int16, metrics over that range against float64,
and the coded size of streams that baseline JPEG cannot code.  Every comparison with the oracle is bit
for bit unless stated otherwise."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from inputs import adversarial
from test_range_cpu import out_of_range_cases, reference_coded_bits, in_range_stream

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

SCALES = [-12, -6, -1, 0, 3, 8, 12, 16]      # s = 2^k: x_s = 128 + s (x0 - 128), Q_s = s Q are exact in f32
BIG = 1e6


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def x0():
    """Integer image, 0..255: the adversarial bands over random blocks, 256 x 256."""
    rng = np.random.default_rng(21)
    img = rng.integers(0, 256, (256, 256)).astype(np.float32)
    adv = adversarial(32)
    img[: adv.shape[0]] = adv
    return img


def scaled(x0, k):
    s = np.float32(2.0 ** k)
    return (np.float32(128) + s * (x0 - np.float32(128))).astype(np.float32), s


def big_image(H, W, seed):
    """f32 pixels up to +-1e6: most quantised coefficients lie far outside int16."""
    rng = np.random.default_rng(seed)
    img = (rng.random((H, W)) * 2 * BIG - BIG).astype(np.float32)
    img[: H // 2, : W // 2] = rng.integers(0, 256, (H // 2, W // 2))      # a quarter that never saturates
    return img


def blocks_any(a, H, W):
    """(H/8, W/8) boolean: any element of the block set."""
    return a.reshape(H // 8, 8, W // 8, 8).any(axis=(1, 3))


# ---------------------------------------------------------------- 1. scale sweep

def forward_paths(dct, oracle):
    T = oracle.dct2_T()
    return {
        "direct": lambda Q: dct.Plan(Q=Q, path=dct.api.PATH_DIRECT),
        "tma": lambda Q: dct.Plan(Q=Q, path=dct.api.PATH_TMA),
        "dense_symmetric": lambda Q: dct.Plan(T=T, Q=Q, dense=dct.api.DENSE_SYMMETRIC),
        "dense_chain": lambda Q: dct.Plan(T=T, Q=Q, dense=dct.api.DENSE_CHAIN),
    }


@pytest.mark.parametrize("path", ["direct", "tma", "dense_symmetric", "dense_chain"])
def test_forward_coefficients_are_scale_invariant(dct, oracle, x0, path):
    """Scaling pixels about 128 and Q by the same power of two leaves every quantised coefficient
    unchanged, bit for bit: the sweep also moves Q from the fast-division kernels (integers up to 255)
    to __fdiv_rn and back."""
    make = forward_paths(dct, oracle)[path]
    Q = oracle.jpeg_Q()
    T = oracle.dct2_T() if path.startswith("dense") else None
    ref = None
    for k in SCALES:
        x, s = scaled(x0, k)
        got = host(dct.forward(dev(x), plan=make(Q * s)))
        if ref is None:
            ref = got
            if path != "dense_symmetric":     # chain order: the oracle's arithmetic
                assert np.array_equal(bits(got), bits(oracle.dct(x0, T=T, Q=Q)))
        assert np.array_equal(bits(got), bits(ref)), f"k={k}"


@pytest.mark.parametrize("path", ["direct", "tma", "dense_chain"])
def test_fused_outputs_equal_the_oracle_at_every_scale(dct, oracle, x0, path):
    """roundtrip (with its coefficient plane), inverse, roundtrip_batch and roundtrip_any at every scale."""
    make = forward_paths(dct, oracle)[path]
    Q = oracle.jpeg_Q()
    T = oracle.dct2_T() if path.startswith("dense") else None
    for k in SCALES:
        x, s = scaled(x0, k)
        plan = make(Q * s)
        want, wcoef = oracle.roundtrip(x, T=T, Q=Q * s, want_coef=True)
        d = dev(x)
        coef = torch.empty_like(d)
        out = dct.roundtrip(d, coef=coef, plan=plan)
        assert np.array_equal(bits(host(out)), bits(want)), f"roundtrip k={k}"
        assert np.array_equal(bits(host(coef)), bits(wcoef)), f"coef k={k}"
        inv = dct.inverse(coef, plan=plan)
        assert np.array_equal(bits(host(inv)), bits(oracle.idct(wcoef, T=T, Q=Q * s))), f"inverse k={k}"
        if path == "tma":
            continue
        outs = dct.roundtrip_batch([d, dev(x[:, ::-1])], plan=plan)
        assert np.array_equal(bits(host(outs[0])), bits(want)), f"batch k={k}"
        assert np.array_equal(bits(host(outs[1])), bits(oracle.roundtrip(np.ascontiguousarray(x[:, ::-1]), T=T, Q=Q * s)))
        xa = np.ascontiguousarray(x[:250, :246])
        got = host(dct.roundtrip_any(dev(xa), plan=plan))
        pad = np.pad(xa, ((0, 6), (0, 2)), mode="edge")
        assert np.array_equal(bits(got), bits(oracle.roundtrip(pad, T=T, Q=Q * s)[:250, :246])), f"any k={k}"


def test_tensor_core_arm_across_scales(dct, oracle, x0):
    """DENSE_MMA: its coefficient plane is the same at every scale (the TF32 hi/lo splits scale with
    the operands), and against the oracle it keeps the arm's own criterion with pixel tolerances scaled."""
    T, Q = oracle.dct2_T(), oracle.jpeg_Q()
    ref = None
    for k in SCALES:
        x, s = scaled(x0, k)
        want, wcoef = oracle.roundtrip(x, T=T, Q=Q * s, want_coef=True)
        d = dev(x)
        coef = torch.empty_like(d)
        out = dct.roundtrip(d, coef=coef, plan=dct.Plan(T=T, Q=Q * s, dense=dct.api.DENSE_MMA))
        assert dct.api.last_path() == "mma"
        gc, go = host(coef), host(out)
        if ref is None:
            ref = gc
        assert np.array_equal(bits(gc), bits(ref)), f"k={k}"
        diff = np.abs(gc - wcoef)
        assert diff.max() <= 1 and np.mean(diff > 0) < 2e-3, (k, diff.max())
        same = diff.reshape(32, 8, 32, 8).max(axis=(1, 3)) == 0
        pix = np.abs(go.astype(np.float64) - want).reshape(32, 8, 32, 8).max(axis=(1, 3))
        assert pix[same].max() < 2e-3 * float(s) + 2.0 ** -16, (k, pix[same].max())


@pytest.mark.parametrize("path", ["direct", "tma"])
def test_negative_quantisers(dct, oracle, x0, path):
    """Q -> -Q negates every coefficient (as values: rounding and masking give signed zeros) and leaves
    the pixels unchanged bit for bit; a mixed-sign table matches the oracle."""
    p = dct.api.PATH_DIRECT if path == "direct" else dct.api.PATH_TMA
    Q = oracle.jpeg_Q()
    d = dev(x0)
    for q in (Q, Q / 8):
        c_pos, c_neg = torch.empty_like(d), torch.empty_like(d)
        o_pos = dct.roundtrip(d, coef=c_pos, plan=dct.Plan(Q=q, path=p))
        o_neg = dct.roundtrip(d, coef=c_neg, plan=dct.Plan(Q=-q, path=p))
        assert np.array_equal(host(c_neg), -host(c_pos))
        assert np.array_equal(bits(host(o_neg)), bits(host(o_pos)))
        f_neg = host(dct.forward(d, plan=dct.Plan(Q=-q, path=p)))
        assert np.array_equal(f_neg, -host(c_pos))
    mixed = (Q * np.where(np.arange(64) % 3 == 0, -1, 1)).astype(np.float32)
    want, wcoef = oracle.roundtrip(x0, Q=mixed, want_coef=True)
    coef = torch.empty_like(d)
    out = dct.roundtrip(d, coef=coef, plan=dct.Plan(Q=mixed, path=p))
    assert np.array_equal(bits(host(out)), bits(want))
    assert np.array_equal(bits(host(coef)), bits(wcoef))


# ---------------------------------------------------------------- 2. saturation

@pytest.mark.parametrize("path", ["direct", "tma"])
def test_forward_saturates_int16_planes(dct, oracle, path):
    H = W = 256
    img = big_image(H, W, 1)
    want = np.clip(oracle.dct(img), -32768, 32767)
    assert (np.abs(oracle.dct(img)) > 32767).mean() > 0.05
    p = dct.api.PATH_DIRECT if path == "direct" else dct.api.PATH_TMA
    d = dev(img)
    c16 = dct.forward(d, plan=dct.Plan(path=p), coef_dtype=torch.int16)
    assert dct.api.last_path() == path
    assert np.array_equal(host(c16).astype(np.float32), want)
    # the zig-zag stream is direct-family only
    zz = dct.forward(d, plan=dct.Plan(path=dct.api.PATH_DIRECT), zigzag=True)
    assert np.array_equal(host(zz), oracle.zigzag_i16(oracle.dct(img)))


@pytest.mark.parametrize("path", ["direct", "tma"])
@pytest.mark.parametrize("coef_kind", ["i16", "zigzag"])
@pytest.mark.parametrize("keep", [0, 6, 8, 10])
def test_fused_round_trip_pixels_ignore_saturation(dct, oracle, path, coef_kind, keep):
    """The coefficient output saturates; the pixels come from the unsaturated coefficients, so an
    inverse of the saturated plane differs from the fused pixels exactly in the blocks that saturated.
    keep = 6..10: the compiled-mask kernels of the default tables."""
    if coef_kind == "zigzag" and path == "tma":
        pytest.skip("zig-zag streams are a direct-family layout")
    H = W = 256
    img = big_image(H, W, 2)
    mask = dct.ALL_COEFFS if keep == 0 else oracle.zigzag_mask(keep)
    want, wcoef = oracle.roundtrip(img, keep=mask, want_coef=True)
    plan = dct.Plan(keep=mask, path=dct.api.PATH_DIRECT if path == "direct" else dct.api.PATH_TMA)
    d = dev(img)
    if coef_kind == "zigzag":
        coef = dct.api.empty_zigzag(H, W, d.device)
        out = dct.roundtrip(d, coef=coef, plan=plan, zigzag=True)
        assert np.array_equal(host(coef), oracle.zigzag_i16(wcoef))
        split = dct.inverse(coef, plan=plan, zigzag=True)
    else:
        coef = torch.empty(H, W, dtype=torch.int16, device="cuda")
        out = dct.roundtrip(d, coef=coef, plan=plan)
        assert np.array_equal(host(coef).astype(np.float32), np.clip(wcoef, -32768, 32767))
        split = dct.inverse(coef, plan=plan)
    assert np.array_equal(bits(host(out)), bits(want))
    saturated = blocks_any(np.abs(wcoef) > 32767, H, W)
    assert saturated.any() and not saturated.all()
    differs = blocks_any(host(split) != host(out), H, W)
    assert np.array_equal(differs, saturated)


@pytest.mark.parametrize("path", ["direct", "tma"])
def test_metrics_with_saturating_coefficients(dct, oracle, path):
    H = W = 256
    img = big_image(H, W, 3)
    want, wcoef = oracle.roundtrip(img, want_coef=True)
    d = dev(img)
    coef = torch.empty(H, W, dtype=torch.int16, device="cuda")
    out, (mse, peen, nnz) = dct.roundtrip_with_metrics(
        d, coef=coef, plan=dct.Plan(path=dct.api.PATH_DIRECT if path == "direct" else dct.api.PATH_TMA))
    assert np.array_equal(host(coef).astype(np.float32), np.clip(wcoef, -32768, 32767))
    assert np.array_equal(bits(host(out)), bits(want))
    assert nnz == int(np.count_nonzero(wcoef))


def extreme_streams(H, W, seed):
    rng = np.random.default_rng(seed)
    c = rng.choice(np.array([32767, -32767, -32768, 0, 1], np.int16), size=(H, W), p=[0.3, 0.3, 0.3, 0.05, 0.05])
    c[:8, :8] = -32768
    c[8:16, :8] = 32767
    return c


@pytest.mark.parametrize("path", ["direct", "tma"])
@pytest.mark.parametrize("kind", ["i16", "zigzag"])
def test_inverse_of_extreme_coefficients(dct, oracle, path, kind):
    if kind == "zigzag" and path == "tma":
        pytest.skip("zig-zag streams are a direct-family layout")
    H = W = 128
    c = extreme_streams(H, W, 5)
    rng = np.random.default_rng(6)
    for Q in (oracle.jpeg_Q() * 2, rng.integers(1, 256, 64).astype(np.float32), np.full(64, 255, np.float32)):
        plan = dct.Plan(Q=Q, path=dct.api.PATH_DIRECT if path == "direct" else dct.api.PATH_TMA)
        want = oracle.idct(c.astype(np.float32), Q=Q)
        src = dev(oracle.zigzag_i16(c.astype(np.float32))) if kind == "zigzag" else dev(c)
        zz = kind == "zigzag"
        got = dct.inverse(src, plan=plan, zigzag=zz)
        assert np.array_equal(bits(host(got)), bits(want))
        got8 = dct.inverse(src, plan=plan, img_dtype=torch.uint8, zigzag=zz)
        assert np.array_equal(host(got8), oracle.to_u8(want))


@pytest.mark.factored
def test_inverse_of_extreme_coefficients_factored(dct, oracle):
    H = W = 128
    c = extreme_streams(H, W, 7)
    for Q in (oracle.jpeg_Q() * 2, np.full(64, 255, np.float32)):
        want = oracle.to_u8(oracle.idct(c.astype(np.float32), Q=Q)).astype(np.int16)
        for p in (dct.api.PATH_DIRECT, dct.api.PATH_TMA):
            got = host(dct.inverse(dev(c), plan=dct.Plan(Q=Q, path=p), img_dtype=torch.uint8)).astype(np.int16)
            assert np.abs(got - want).max() <= 1


def worst_case_rgb(H, W):
    """Flat 0, flat 255 and +-128 basis patterns per channel, so that every plane reaches its extremes."""
    yy, xx = np.mgrid[0:H, 0:W]
    rgb = np.zeros((H, W, 3), np.int32)
    band = (yy // 8) % 6
    pat = np.where(((xx + yy) % 2) == 0, 255, 0)
    rgb[band == 1] = 255
    for c in range(3):
        rgb[..., c] = np.where(band == 2, pat if c != 1 else 255 - pat, rgb[..., c])
        rgb[..., c] = np.where(band == 3, np.where((xx // 4) % 2 == c % 2, 255, 0), rgb[..., c])
        rgb[..., c] = np.where(band == 4, np.where((yy // 4) % 2 == c % 2, 0, 255), rgb[..., c])
    rng = np.random.default_rng(9)
    rgb[band == 5] = rng.integers(0, 256, (int((band == 5).sum()), 3))
    return rgb.astype(np.uint8)


def test_rgb_split_at_the_documented_floor(dct, oracle):
    """Every Q entry 1/16: no stream value saturates and the split call is the fused call."""
    H, W = 96, 128
    rgb = worst_case_rgb(H, W)
    q = np.full(64, 1 / 16, np.float32)
    plan = dct.Plan(Q=q, Qc=q, inverse=dct.api.INVERSE_EXACT)
    d = dev(rgb)
    zz = dct.forward_rgb(d, plan=plan)
    assert int(np.abs(host(zz).astype(np.int32)).max()) < 32767
    assert torch.equal(dct.inverse_rgb(zz, plan=plan), dct.roundtrip_rgb(d, plan=plan))


def test_rgb_beyond_the_documented_floor(dct, oracle):
    """Every Q entry 1/64: the streams are the oracle's saturated streams; the fused pixels still equal
    the oracle's, computed from the unsaturated coefficients."""
    H, W = 96, 128
    rgb = worst_case_rgb(H, W)
    q = np.full(64, 1 / 64, np.float32)
    plan = dct.Plan(Q=q, Qc=q, inverse=dct.api.INVERSE_EXACT)
    want, _, coef3 = oracle.roundtrip_rgb(rgb, Q=q, Qc=q, want_planes=True, want_coef=True)
    assert (np.abs(coef3) > 32767).any()
    d = dev(rgb)
    zz = host(dct.forward_rgb(d, plan=plan))
    for c in range(3):
        assert np.array_equal(zz[c], oracle.zigzag_i16(coef3[c])), c
    streams = torch.empty(3, H // 8, W // 8, 64, dtype=torch.int16, device="cuda")
    fused = dct.roundtrip_rgb(d, streams=streams, plan=plan)
    assert np.array_equal(host(fused), want)
    assert np.array_equal(host(streams), zz)


# ---------------------------------------------------------------- 3. metrics over the range

def metrics_case(name, N, oracle):
    rng = np.random.default_rng(N)
    yy, xx = np.mgrid[0:N, 0:N].astype(np.float32)
    smooth = (0.5 + 0.4 * np.sin(xx / 17.0) * np.cos(yy / 23.0) + 0.02 * rng.standard_normal((N, N))).astype(np.float32)
    Q = oracle.jpeg_Q()
    if name == "8bit":
        return np.round(smooth * 255).astype(np.float32), Q
    if name == "unit_q255":
        return smooth, (Q / 255).astype(np.float32)
    if name == "unit_q4096":                          # near lossless
        return smooth, (Q / 4096).astype(np.float32)
    if name == "tiny":                                # pixels ~2^-10
        return (smooth * 2.0 ** -10).astype(np.float32), (Q * 2.0 ** -18).astype(np.float32)
    if name == "u16":
        return np.round(smooth * 65535).astype(np.float32), (Q * 256).astype(np.float32)
    if name == "huge":                                # pixels up to 2^20
        return np.round(smooth * 2.0 ** 20).astype(np.float32), (Q * 4096).astype(np.float32)
    raise KeyError(name)


def f64_metrics(x, y):
    d = x.astype(np.float64) - y.astype(np.float64)
    sse, en = float(np.sum(d * d)), float(np.sum(x.astype(np.float64) ** 2))
    return sse / x.size, 100.0 * (sse / en) ** 0.5


@pytest.mark.parametrize("N", [256, 2048, 4096])
@pytest.mark.parametrize("name", ["8bit", "unit_q255", "unit_q4096", "tiny", "u16", "huge"])
def test_fused_metrics_against_float64(dct, oracle, N, name):
    """Both one-launch forms (TMA metrics kernel, direct family's) and b200dct_metrics_accumulate:
    within 1e-6 of float64 on the kernel's own input and output, the same bits run to run and on
    both families, and the exact non-zero count."""
    x, Q = metrics_case(name, N, oracle)
    want, wcoef = oracle.roundtrip(x, Q=Q, want_coef=True, threads=oracle.max_threads())
    d = dev(x)
    results = {}
    for fam, p in (("tma", dct.api.PATH_TMA), ("direct", dct.api.PATH_DIRECT)):
        plan = dct.Plan(Q=Q, path=p)
        runs = []
        for _ in range(2):
            out, m = dct.roundtrip_with_metrics(d, plan=plan)
            assert dct.api.last_path() == fam and dct.api.last_launch_count() == 1
            runs.append(m)
        assert runs[0] == runs[1], (fam, runs)
        y = host(out)
        assert np.array_equal(bits(y), bits(want))
        mse, peen = f64_metrics(x, y)
        assert abs(runs[0][0] - mse) <= 1e-6 * mse, (fam, runs[0][0], mse)
        assert abs(runs[0][1] - peen) <= 1e-6 * peen, (fam, runs[0][1], peen)
        assert runs[0][2] == int(np.count_nonzero(wcoef))
        results[fam] = runs[0]
    assert results["tma"] == results["direct"]
    yt = dev(want)
    mse_a, peen_a = dct.metrics(d, yt)
    mse, peen = f64_metrics(x, want)
    assert abs(mse_a - mse) <= 1e-6 * mse and abs(peen_a - peen) <= 1e-6 * peen


# ---------------------------------------------------------------- 4. coded size

def raw_coded_bits(dct, zz, table):
    """b200dct_zigzag_coded_bits through the C ABI: the 64-bit word with its flag."""
    p, _, pitch, H, W = dct.api._zz_plane(zz)
    acc = torch.zeros(1, dtype=torch.int64, device="cuda")
    rc = dct.lib().b200dct_zigzag_coded_bits(p, pitch, H, W, table, acc.data_ptr(),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    return int(acc.item()) & ((1 << 64) - 1)


@pytest.mark.parametrize("table", [0, 1])
def test_coded_bits_in_range_extremes(dct, oracle, table):
    s = in_range_stream(32 * 24, 11).reshape(32, 24, 64)
    want, flag = reference_coded_bits(s, table, oracle)
    assert not flag
    assert raw_coded_bits(dct, dev(s), table) == want == oracle.coded_bits(s, table)
    assert dct.coded_bits(dev(s), table) == want


@pytest.mark.parametrize("table", [0, 1])
@pytest.mark.parametrize("case", range(6))
def test_coded_bits_flag_out_of_range_symbols(dct, oracle, table, case):
    name, s = out_of_range_cases()[case]
    s = s.reshape(2, 2, 64)
    got = raw_coded_bits(dct, dev(s), table)
    assert got == oracle.coded_bits(s, table), name
    assert got >> 63 == 1, name
    with pytest.raises(dct.B200DCTError):
        dct.coded_bits(dev(s), table)
    with pytest.raises(dct.B200DCTError):
        dct.compression_factor(dev(s), table)


def test_coded_bits_flag_on_a_real_stream_and_a_padded_one(dct, oracle):
    """forward(..., zigzag=True) at every Q entry 1/16 on 8-bit content, stored as is and inside a
    wider (pitched) buffer whose padding holds only zeros."""
    img = oracle.rand_image(64, 96, 13)
    q = np.full(64, 1 / 16, np.float32)
    zz = dct.forward(dev(img), plan=dct.Plan(Q=q, path=dct.api.PATH_DIRECT), zigzag=True)
    want = oracle.coded_bits(oracle.zigzag_i16(oracle.dct(img, Q=q)), 0)
    assert want >> 63 == 1
    assert raw_coded_bits(dct, zz, 0) == want
    wide = torch.zeros(8, 12 + 5, 64, dtype=torch.int16, device="cuda")
    wide[:, :12] = zz
    assert raw_coded_bits(dct, wide[:, :12], 0) == want
    # a padded in-range stream: the padding is not read
    ok = dev(in_range_stream(8 * 12, 3).reshape(8, 12, 64))
    wide.fill_(-32768)
    wide[:, :12] = ok
    assert raw_coded_bits(dct, wide[:, :12], 1) == oracle.coded_bits(host(ok), 1) < 1 << 63
