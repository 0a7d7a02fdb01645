"""CPU suite: the oracle against its fixtures, known answers and size-independent
properties.  No GPU.  (The oracle is test infrastructure; see oracle/dct_oracle.c.)"""
import glob
import os

import numpy as np
import pytest

import inputs

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_constants_bit_patterns(oracle):
    # SURVEY.md Appendix A.1: the f32 bit patterns of the reference's double literals
    T = oracle.haweel_T().view(np.uint32)
    assert T[0] == 0x3EB504F3 and T[8] == 0x3F000000 and T[16] == 0x3EE4F92E
    assert T[17] == 0x3E64F92E and T[29] == 0x3F3504F3 and T[26] == 0xBF3504F3
    assert np.count_nonzero(oracle.haweel_T()) == 44
    Q = oracle.jpeg_Q()
    assert Q.min() == 10 and Q.max() == 121 and len(set(Q.tolist())) == 47
    # Haweel's T is orthogonal up to f32 rounding
    T2 = oracle.haweel_T().reshape(8, 8).astype(np.float64)
    assert np.abs(T2 @ T2.T - np.eye(8)).max() < 1e-6


@pytest.mark.parametrize("N,s,sa,nz,su8,mse,peen", [
    # SURVEY.md Appendix B (reference generator srand(42), rand()%256)
    (256, -306, 114414, 46317, 8329775, 342.731643677, 12.552802314),
    (1024, -2562, 1831230, 741557, 133161285, 344.862137794, 12.604274134),
    (8192, -268447, 117045095, 47462419, 8524699637, 344.379744306, 12.593068395),   # the headline size
])
def test_known_answers(oracle, N, s, sa, nz, su8, mse, peen):
    img = oracle.rand_image(N, N, 42)
    out, coef = oracle.roundtrip(img, want_coef=True, threads=max(1, min(8, os.cpu_count() or 1)))
    assert int(coef.sum(dtype=np.float64)) == s
    assert int(np.abs(coef).sum(dtype=np.float64)) == sa
    assert int(np.count_nonzero(coef)) == nz
    u8 = oracle.to_u8(out)
    assert int(u8.sum(dtype=np.int64)) == su8
    m, p = oracle.metrics(img.astype(np.uint8), u8)
    assert m == pytest.approx(mse, rel=1e-9) and p == pytest.approx(peen, rel=1e-9)


def test_known_block(oracle):
    # SURVEY.md Appendix B: block (0,0) of the 256x256 reference input
    img = oracle.rand_image(256, 256, 42)
    assert img[0, :8].tolist() == [70, 100, 49, 41, 100, 134, 237, 156]
    coef = oracle.dct(img)
    assert coef[:8, :8].astype(int).tolist()[0] == [4, -3, -3, -2, -4, 2, -2, 2]
    assert coef[:8, 0].astype(int).tolist() == [4, 7, -8, -7, -10, -1, 2, -3]
    rec = oracle.idct(coef)
    np.testing.assert_allclose(rec[0, :8], [85.6244, 105.1761, 74.1841, 36.4329, 93.9596, 136.4364, 229.7527, 151.5972], atol=1e-3)
    assert rec[:8, :8].min() < 0 and rec[:8, :8].max() > 255  # both clamps exercised


def test_golden_fixtures(oracle):
    g = np.load(os.path.join(GOLD, "oracle_rand256.npz"))
    out, coef = oracle.roundtrip(g["img"].astype(np.float32), want_coef=True)
    assert np.array_equal(coef.astype(np.int16), g["coef"])
    assert np.array_equal(out.view(np.uint32), g["out"].view(np.uint32))
    assert np.array_equal(oracle.to_u8(out), g["out_u8"])
    g = np.load(os.path.join(GOLD, "oracle_adversarial.npz"))
    assert np.array_equal(g["img"], inputs.adversarial(16).astype(np.uint8))
    out, coef = oracle.roundtrip(g["img"].astype(np.float32), want_coef=True)
    assert np.array_equal(coef.astype(np.int16), g["coef"])
    assert np.array_equal(out.view(np.uint32), g["out"].view(np.uint32))
    g = np.load(os.path.join(GOLD, "oracle_masks.npz"))
    for k in (6, 7, 8, 9, 10):
        out, coef = oracle.roundtrip(g["img"].astype(np.float32), keep=oracle.zigzag_mask(k), want_coef=True)
        assert np.array_equal(coef.astype(np.int16), g[f"coef_k{k}"])
        assert np.array_equal(out.view(np.uint32), g[f"out_k{k}"].view(np.uint32))
    g = np.load(os.path.join(GOLD, "oracle_dense_dct2.npz"))
    out, coef = oracle.roundtrip(g["img"].astype(np.float32), T=g["T"], want_coef=True)
    assert np.array_equal(coef.astype(np.int16), g["coef"])
    assert np.array_equal(out.view(np.uint32), g["out"].view(np.uint32))


def test_reference_gpu_fixtures(oracle):
    """Fixtures written on the B200 box by the UNMODIFIED reference kernels
    (tests/golden/make_ref_golden.py): they pin the CPU restatement to the reference."""
    files = sorted(glob.glob(os.path.join(GOLD, "refgpu_*.npz")))
    if not files:
        pytest.skip("no refgpu_*.npz committed yet (generated on the GPU box)")
    for f in files:
        g = np.load(f)
        img = g["img"].astype(np.float32)
        coef, shifted = oracle.dct(img, want_shifted=True)
        assert np.array_equal(coef.view(np.uint32), g["coef"].view(np.uint32)), f
        assert np.array_equal(shifted, g["shifted"]), f
        rec = oracle.idct(coef)
        assert np.array_equal(rec.view(np.uint32), g["rec"].view(np.uint32)), f


def test_stored_oracle_digests_are_still_reproduced(oracle):
    """tests/golden/refgpu_digests.json (the oracle's digests, which the GPU suite compares with
    where the reference is not built) is still what the oracle produces, on its smaller cases.
    A guard against changes of the oracle or edits of the file; what pins the oracle to the
    reference is test_reference_gpu_fixtures."""
    import refgpu

    for case, img, Q in (("rand256", oracle.rand_image(256, 256, 42), None), ("adversarial32", inputs.adversarial(32), None),
                         ("floatnoise64x256", inputs.float_noise(64, 256), None),
                         ("rand256_seed5_halfq", oracle.rand_image(256, 256, 5), oracle.jpeg_Q() * 0.5)):
        want = refgpu.stored(case)
        coef, shifted = oracle.dct(img, Q=Q, want_shifted=True)
        assert refgpu.digest(coef) == want["coef"] and refgpu.digest(shifted) == want["shifted"], case
        assert refgpu.digest(oracle.idct(coef, Q=Q)) == want["rec"], case


def test_split_equals_fused_and_u8(oracle):
    img = inputs.adversarial(8)
    coef = oracle.dct(img)
    rec = oracle.idct(coef)
    out, coef2 = oracle.roundtrip(img, want_coef=True)
    assert np.array_equal(coef.view(np.uint32), coef2.view(np.uint32))
    assert np.array_equal(rec.view(np.uint32), out.view(np.uint32))
    u8 = img.astype(np.uint8)
    out8, coef8 = oracle.roundtrip(u8, want_coef=True)
    assert np.array_equal(coef8, coef)
    assert np.array_equal(out8, oracle.to_u8(rec))


def test_u8_conversion_edges(oracle):
    v = np.array([-5.0, -0.0, 0.0, 0.999, 1.0, 254.999, 255.0, 255.5, 300.0, 127.5, np.nextafter(np.float32(256), np.float32(0))], np.float32)
    assert oracle.to_u8(v).tolist() == [0, 0, 0, 0, 1, 254, 255, 255, 255, 127, 255]


def test_block_independence_and_stripes(oracle):
    # a stripe of block-rows transforms to the same rows of the full-image result
    img = oracle.rand_image(64, 96, 3)
    full = oracle.roundtrip(img)
    for r0, r1 in ((0, 8), (8, 40), (40, 64)):
        part = oracle.roundtrip(np.ascontiguousarray(img[r0:r1]))
        assert np.array_equal(part.view(np.uint32), full[r0:r1].view(np.uint32))
    # a batch stored back to back is one tall image
    a, b = oracle.rand_image(16, 32, 1), oracle.rand_image(16, 32, 2)
    both = oracle.roundtrip(np.concatenate([a, b]))
    assert np.array_equal(both[:16], oracle.roundtrip(a)) and np.array_equal(both[16:], oracle.roundtrip(b))


def test_mask_semantics(oracle):
    assert oracle.zigzag_mask(0) == 0 and oracle.zigzag_mask(64) == (1 << 64) - 1
    # first ten zig-zag positions (row, col), SURVEY.md section 8c
    want = [(0, 0), (0, 1), (1, 0), (2, 0), (1, 1), (0, 2), (0, 3), (1, 2), (2, 1), (3, 0)]
    for k in range(1, 11):
        m = oracle.zigzag_mask(k)
        assert {(i // 8, i % 8) for i in range(64) if (m >> i) & 1} == set(want[:k])
    img = oracle.rand_image(32, 32, 5)
    full = oracle.dct(img)
    for k in (1, 6, 10, 64):
        m = oracle.zigzag_mask(k)
        c = oracle.dct(img, keep=m)
        keepmat = np.array([(m >> i) & 1 for i in range(64)], bool).reshape(8, 8)
        tiled = np.tile(keepmat, (4, 4))
        assert np.array_equal(c[tiled], full[tiled]) and not c[~tiled].any()
        # masked round trip == reference dct -> host zeroing -> reference idct
        assert np.array_equal(oracle.roundtrip(img, keep=m), oracle.idct(np.where(tiled, full, 0).astype(np.float32)))
    # keeping more coefficients never increases the error on a smooth image
    sm = inputs.smooth_image(64, 64)
    errs = [oracle.metrics(sm, oracle.roundtrip(sm, keep=oracle.zigzag_mask(k)))[0] for k in (6, 10, 64)]
    assert errs[0] >= errs[1] >= errs[2]


def test_linearity_of_unquantised_transform(oracle):
    # with Q = 1 and tiny inputs nothing rounds to a different integer: check orthogonality
    # through the public behaviour: constant block -> only DC, value 8*(v-128)/Q00
    img = np.full((8, 8), 160.0, np.float32)
    c = oracle.dct(img)
    assert c[0, 0] == round(8 * 32 / 16) and not c.reshape(-1)[1:].any()


def test_idempotent_requantisation(oracle):
    # quantise(dequantise(C)) == C: forward of an exactly reconstructed block returns the
    # same coefficients when the reconstruction is not clamped (dense orthonormal DCT-II)
    T = oracle.dct2_T()
    img = inputs.smooth_image(32, 32)
    c1 = oracle.dct(img, T=T)
    rec = oracle.idct(c1, T=T)
    c2 = oracle.dct(rec, T=T)
    assert np.abs(c1 - c2).max() <= 1  # rounding of the f32 reconstruction may move a tie
    assert (c1 != c2).mean() < 0.01


def test_metrics_definition(oracle):
    x = np.array([[10, 20], [30, 40]], np.uint8)
    y = np.array([[11, 18], [30, 44]], np.uint8)
    mse, peen = oracle.metrics(x, y)
    assert mse == pytest.approx((1 + 4 + 0 + 16) / 4)
    assert peen == pytest.approx(100 * np.sqrt(21 / 3000))


def test_multithreaded_oracle_matches_sequential(oracle):
    img = oracle.rand_image(128, 128, 9)
    assert np.array_equal(oracle.roundtrip(img, threads=1), oracle.roundtrip(img, threads=4))


def test_zigzag_stream_layout(oracle):
    """The zig-zag scan of the compact coefficient stream is ITU-T T.81's: regenerate it by
    walking the anti-diagonals and compare; round trip through the stream is lossless for
    coefficients in int16 range and saturates outside."""
    order = []
    for s in range(15):
        diag = [(r, s - r) for r in range(8) if 0 <= s - r < 8]
        order += diag if s % 2 else diag[::-1]  # even diagonals run bottom-left -> top-right
    plane = np.arange(64, dtype=np.float32).reshape(8, 8)
    assert oracle.zigzag_i16(plane)[0, 0].tolist() == [r * 8 + c for r, c in order]
    assert [bin(oracle.zigzag_mask(k)).count("1") for k in (6, 10)] == [6, 10]
    img = oracle.rand_image(16, 24, 3)
    coef = oracle.dct(img)
    zz = oracle.zigzag_i16(coef)
    assert zz.shape == (2, 3, 64)
    assert np.array_equal(oracle.unzigzag_i16(zz), coef)
    assert zz[1, 2, 0] == coef[8, 16] and zz[1, 2, 1] == coef[8, 17] and zz[1, 2, 2] == coef[9, 16]
    big = np.full((8, 8), 1e6, np.float32); big[0, 1] = -1e6
    assert oracle.zigzag_i16(big)[0, 0, :2].tolist() == [32767, -32768]
