"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs.  Tolerances: quantised coefficients and f32/u8 pixels are compared BIT-EXACT (the
kernels reproduce the reference's FMA chains, so the +-1 LSB allowance of the spec is not
needed); MSE/PEEN to 1e-9 relative (spec: 1e-3)."""
import numpy as np
import pytest
import torch

import inputs

pytestmark = pytest.mark.gpu

PATHS = {"tma": 2, "direct": 1}


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


@pytest.mark.parametrize("path", ["tma", "direct"])
@pytest.mark.parametrize("shape", [(8, 32), (256, 256), (64, 96), (1024, 1024), (520, 2048 + 32)])
def test_roundtrip_f32_bit_exact(dct, oracle, path, shape):
    img = oracle.rand_image(*shape, 42)
    want_out, want_coef = oracle.roundtrip(img, want_coef=True)
    plan = dct.Plan(path=PATHS[path])
    d = dev(img)
    coef = torch.empty_like(d)
    out = dct.roundtrip(d, coef=coef, plan=plan)
    assert dct.api.last_path() == path
    assert np.array_equal(bits(host(coef)), bits(want_coef))
    assert np.array_equal(bits(host(out)), bits(want_out))
    assert np.array_equal(host(d), img)  # the fused entry point does not touch its input
    out2 = dct.roundtrip(d, plan=plan)   # without the coefficient plane
    assert np.array_equal(bits(host(out2)), bits(want_out))


@pytest.mark.parametrize("path", ["tma", "direct"])
def test_split_forward_inverse(dct, oracle, path):
    img = inputs.adversarial(32)  # 256 wide
    want_coef, want_shift = oracle.dct(img, want_shifted=True)
    want_rec = oracle.idct(want_coef)
    plan = dct.Plan(path=PATHS[path])
    coef = dct.forward(dev(img), plan=plan)
    assert np.array_equal(bits(host(coef)), bits(want_coef))
    rec = dct.inverse(coef, plan=plan)
    assert np.array_equal(bits(host(rec)), bits(want_rec))
    # compact int16 coefficients carry the same integers
    c16 = dct.forward(dev(img), plan=plan, coef_dtype=torch.int16)
    assert np.array_equal(host(c16), want_coef.astype(np.int16))
    rec16 = dct.inverse(c16, plan=plan)
    assert np.array_equal(bits(host(rec16)), bits(oracle.idct(want_coef.astype(np.int16).astype(np.float32))))
    # u8 output of the inverse = convertToUnsignedChar
    rec8 = dct.inverse(coef, plan=plan, img_dtype=torch.uint8)
    assert np.array_equal(host(rec8), oracle.to_u8(want_rec))


def test_forward_side_effect_shifted(dct, oracle):
    img = oracle.rand_image(64, 64, 1)
    want_coef, want_shift = oracle.dct(img, want_shifted=True)
    d = dev(img)
    coef = dct.forward(d, shifted=d)  # in place, as the reference's sub_matrix_scalar
    assert np.array_equal(bits(host(coef)), bits(want_coef))
    assert np.array_equal(host(d), want_shift)


@pytest.mark.parametrize("path", ["tma", "direct"])
@pytest.mark.parametrize("shape", [(8, 32), (256, 256), (72, 1056)])
def test_roundtrip_u8(dct, oracle, path, shape):
    img = oracle.rand_image_u8(*shape, 42)
    want_out, want_coef = oracle.roundtrip(img, want_coef=True)
    plan = dct.Plan(path=PATHS[path])
    coef = torch.empty(shape, dtype=torch.float32, device="cuda")
    out = dct.roundtrip(dev(img), coef=coef, plan=plan)
    assert dct.api.last_path() == path
    assert np.array_equal(host(out), want_out)
    assert np.array_equal(bits(host(coef)), bits(want_coef))
    c16 = torch.empty(shape, dtype=torch.int16, device="cuda")
    out = dct.roundtrip(dev(img), coef=c16, plan=plan)
    assert np.array_equal(host(out), want_out) and np.array_equal(host(c16), want_coef.astype(np.int16))
    c = dct.forward(dev(img), plan=plan)
    assert np.array_equal(bits(host(c)), bits(want_coef))


def test_auto_path_policy(dct, oracle):
    """AUTO: the TMA family for large HBM-bound sparse-T calls, the direct family otherwise."""
    small = torch.zeros(256, 256, device="cuda")
    big = torch.zeros(6144, 6144, device="cuda")
    dct.roundtrip(small)
    assert dct.api.last_path() == "direct"
    dct.roundtrip(big)
    assert dct.api.last_path() == "tma"
    dct.forward(big)
    assert dct.api.last_path() == "tma"
    dct.roundtrip(big.to(torch.uint8))
    assert dct.api.last_path() == "direct"          # 2 B/px: FP32-pipe bound
    dct.roundtrip(big, plan=dct.Plan(T=oracle.dct2_T()))
    assert dct.api.last_path() == "direct"          # dense T: FP32-pipe bound
    dct.roundtrip(big.to(torch.uint8), coef=torch.empty(6144, 6144, device="cuda"))
    assert dct.api.last_path() == "tma"             # + f32 coefficient plane: 6 B/px


@pytest.mark.parametrize("shape", [(8, 8), (8, 16), (72, 1040), (16, 24)])
def test_auto_path_falls_back_to_direct_on_narrow_or_odd_widths(dct, oracle, shape):
    """W % 32 != 0 cannot be tiled by the f32 TMA view: AUTO silently uses the direct kernels,
    forcing TMA is an error (never a wrong result)."""
    img8 = oracle.rand_image_u8(*shape, 42)
    img = img8.astype(np.float32)
    want_out, want_coef = oracle.roundtrip(img, want_coef=True)
    coef = torch.empty(shape, dtype=torch.float32, device="cuda")
    out = dct.roundtrip(dev(img), coef=coef)
    assert dct.api.last_path() == "direct"
    assert np.array_equal(bits(host(out)), bits(want_out)) and np.array_equal(bits(host(coef)), bits(want_coef))
    assert np.array_equal(host(dct.roundtrip(dev(img8))), oracle.to_u8(want_out))
    with pytest.raises(dct.B200DCTError):
        dct.roundtrip(dev(img), plan=dct.Plan(path=2))


@pytest.mark.parametrize("path", ["tma", "direct"])
def test_adversarial_and_float_inputs(dct, oracle, path):
    plan = dct.Plan(path=PATHS[path])
    for img in (inputs.adversarial(32), inputs.float_noise(64, 256), inputs.smooth_image(128, 128),
                np.full((8, 32), -1e4, np.float32), np.full((8, 32), 3e5, np.float32)):
        want_out, want_coef = oracle.roundtrip(img, want_coef=True)
        coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
        out = dct.roundtrip(dev(img), coef=coef, plan=plan)
        assert np.array_equal(bits(host(coef)), bits(want_coef))
        assert np.array_equal(bits(host(out)), bits(want_out))


@pytest.mark.parametrize("path", ["tma", "direct"])
@pytest.mark.parametrize("k", [0, 1, 6, 7, 8, 9, 10, 63])
def test_retained_coefficient_mask(dct, oracle, path, k):
    img = oracle.rand_image(64, 64, 11)
    keep = oracle.zigzag_mask(k)
    want_out, want_coef = oracle.roundtrip(img, keep=keep, want_coef=True)
    plan = dct.Plan(keep=keep, path=PATHS[path])
    coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
    out = dct.roundtrip(dev(img), coef=coef, plan=plan)
    assert np.array_equal(bits(host(coef)), bits(want_coef))
    assert np.array_equal(bits(host(out)), bits(want_out))
    u8 = img.astype(np.uint8)
    assert np.array_equal(host(dct.roundtrip(dev(u8), plan=plan)), oracle.roundtrip(u8, keep=keep))


@pytest.mark.parametrize("path", ["tma", "direct"])
def test_custom_quant_tables(dct, oracle, path):
    img = oracle.rand_image(64, 64, 12)
    for Q in (np.ones(64, np.float32), oracle.jpeg_Q() * 2, np.arange(1, 65, dtype=np.float32),
              oracle.jpeg_Q() * 0.37, np.full(64, 255.0, np.float32)):   # 0.37*Q: not integers -> exact-division kernels
        want_out, want_coef = oracle.roundtrip(img, Q=Q, want_coef=True)
        plan = dct.Plan(Q=Q, path=PATHS[path])
        coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
        out = dct.roundtrip(dev(img), coef=coef, plan=plan)
        assert np.array_equal(bits(host(coef)), bits(want_coef))
        assert np.array_equal(bits(host(out)), bits(want_out))


@pytest.mark.parametrize("path", ["tma", "direct"])
def test_dense_transform_exact_dct(dct, oracle, path):
    """The "exact DCT" variants: any dense 8x8 T as data (SURVEY.md S3)."""
    rng = np.random.default_rng(0)
    for T in (oracle.dct2_T(), rng.standard_normal(64).astype(np.float32) * 0.4):
        img = oracle.rand_image(64, 128, 13)
        want_out, want_coef = oracle.roundtrip(img, T=T, want_coef=True)
        plan = dct.Plan(T=T, path=PATHS[path])
        assert not plan.is_sparse
        coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
        out = dct.roundtrip(dev(img), coef=coef, plan=plan)
        assert np.array_equal(bits(host(coef)), bits(want_coef))
        assert np.array_equal(bits(host(out)), bits(want_out))
        c = dct.forward(dev(img), plan=plan)
        assert np.array_equal(bits(host(c)), bits(want_coef))
        assert np.array_equal(bits(host(dct.inverse(c, plan=plan))), bits(want_out))
        u8 = img.astype(np.uint8)
        assert np.array_equal(host(dct.roundtrip(dev(u8), plan=plan)), oracle.roundtrip(u8, T=T))
    # a dense plan fed Haweel's matrix takes the sparse kernels and gives the same bits
    assert dct.Plan(T=oracle.haweel_T()).is_sparse


def test_golden_fixtures_on_gpu(dct, oracle):
    import os

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_rand256.npz"))
    coef = torch.empty((256, 256), dtype=torch.int16, device="cuda")
    out = dct.roundtrip(dev(g["img"].astype(np.float32)), coef=coef)
    assert np.array_equal(host(coef), g["coef"]) and np.array_equal(bits(host(out)), bits(g["out"]))
    assert np.array_equal(host(dct.roundtrip(dev(g["img"]))), g["out_u8"])


def test_pitched_views_and_batches(dct, oracle):
    img = oracle.rand_image(64, 256, 21)
    big = torch.zeros(64, 512, device="cuda")
    big[:, 128:384] = dev(img)
    view = big[:, 128:384]            # pitch 2048 B, offset 512 B
    out = dct.roundtrip(view)
    assert np.array_equal(bits(host(out)), bits(oracle.roundtrip(img)))
    outv = torch.zeros(64, 512, device="cuda")
    dct.roundtrip(view, out=outv[:, 256:512])
    assert np.array_equal(bits(host(outv[:, 256:512].contiguous())), bits(oracle.roundtrip(img)))
    assert not host(outv[:, :256]).any()   # nothing written outside the destination view
    batch = np.stack([oracle.rand_image(32, 64, s) for s in (1, 2, 3)])
    ob = dct.roundtrip(dev(batch))
    for i in range(3):
        assert np.array_equal(bits(host(ob)[i]), bits(oracle.roundtrip(batch[i])))
    # misaligned sub-view (offset 4 B) is refused, not silently mis-read
    with pytest.raises(dct.B200DCTError):
        dct.roundtrip(big[:, 1:257])
    with pytest.raises(dct.B200DCTError):
        dct.roundtrip(torch.zeros(12, 32, device="cuda"))


def test_host_roundtrip_and_metrics(dct, oracle):
    img = oracle.rand_image(1024, 512, 5)
    want = oracle.roundtrip(img)
    assert np.array_equal(bits(dct.roundtrip_host(img)), bits(want))
    u8 = img.astype(np.uint8)
    want8 = oracle.roundtrip(u8)
    pinned = torch.from_numpy(u8).pin_memory()
    got8 = dct.roundtrip_host(pinned)
    assert np.array_equal(got8.numpy(), want8)
    mse, peen = dct.metrics(dev(u8), dev(want8))
    wm, wp = oracle.metrics(u8, want8)
    assert mse == pytest.approx(wm, rel=1e-9) and peen == pytest.approx(wp, rel=1e-9)
    mse, peen = dct.metrics(dev(img), dev(want))
    wm, wp = oracle.metrics(img, want)
    assert mse == pytest.approx(wm, rel=1e-9) and peen == pytest.approx(wp, rel=1e-9)


@pytest.mark.parametrize("shape", [(8, 8), (256, 256), (72, 1040), (1024, 2048)])
def test_fused_metrics(dct, oracle, shape):
    """b200dct_roundtrip_metrics: pixels identical to the plain round trip; MSE/PEEN equal the
    oracle's double-precision values (u8: exactly, the in-kernel sums are integers;
    f32: to 1e-6 relative, the in-kernel per-block sums are float) -- spec tolerance is 1e-3;
    non-zero count equals the coefficient plane's."""
    img8 = oracle.rand_image_u8(*shape, 7)
    want8, wcoef = oracle.roundtrip(img8, want_coef=True)
    out8, (mse, peen, nnz) = dct.roundtrip_with_metrics(dev(img8))
    assert np.array_equal(host(out8), want8)
    wm, wp = oracle.metrics(img8, want8)
    assert mse == pytest.approx(wm, rel=1e-13) and peen == pytest.approx(wp, rel=1e-13)
    assert nnz == int(np.count_nonzero(wcoef))
    img = inputs.float_noise(*shape, seed=3)
    want, wcoef = oracle.roundtrip(img, want_coef=True)
    coef = torch.empty(shape, dtype=torch.int16, device="cuda")
    out, (mse, peen, nnz) = dct.roundtrip_with_metrics(dev(img), coef=coef, plan=dct.Plan(keep=oracle.zigzag_mask(10)))
    want, wcoef = oracle.roundtrip(img, keep=oracle.zigzag_mask(10), want_coef=True)
    assert np.array_equal(bits(host(out)), bits(want)) and np.array_equal(host(coef), wcoef.astype(np.int16))
    wm, wp = oracle.metrics(img, want)
    assert mse == pytest.approx(wm, rel=1e-6) and peen == pytest.approx(wp, rel=1e-6)
    assert nnz == int(np.count_nonzero(wcoef))
    with pytest.raises(dct.B200DCTError):
        x = dev(img)
        dct.roundtrip_with_metrics(x, out=x)      # aliasing would corrupt the comparison


def test_reference_named_entry_points(dct, oracle):
    """dct_all_blocks_cuda / idct_all_blocks_cuda with the reference's calling convention:
    (image, H, W, T_device, result), input left holding image-128."""
    img = oracle.rand_image(48, 80, 3)   # rectangular: rows=48, cols=80
    want_coef, want_shift = oracle.dct(img, want_shifted=True)
    d_img, T = dev(img), dev(oracle.haweel_T())
    coef, rec = torch.empty_like(d_img), torch.empty_like(d_img)
    dct.api.compat_lib().b200dct_compat_set_options(1, 0)
    dct.dct_all_blocks_cuda(d_img, 48, 80, T, coef)
    assert np.array_equal(bits(host(coef)), bits(want_coef))
    assert np.array_equal(host(d_img), want_shift)
    dct.idct_all_blocks_cuda(coef, 48, 80, T, rec)
    assert np.array_equal(bits(host(rec)), bits(oracle.idct(want_coef)))
    # the cuBLAS-named variants with a dense DCT-II matrix, v2's in-place dequantisation
    T2 = oracle.dct2_T()
    d_img = dev(img)
    dct.dct_all_blocks(d_img, 48, 80, dev(T2), coef, None)
    wc = oracle.dct(img, T=T2)
    assert np.array_equal(bits(host(coef)), bits(wc))
    keep = coef.clone()
    dct.idct_all_blocks(coef, 48, 80, dev(T2), rec, None, dequant_in_place=True)
    assert np.array_equal(bits(host(rec)), bits(oracle.idct(wc, T=T2)))
    assert np.array_equal(host(coef), host(keep) * np.tile(oracle.jpeg_Q().reshape(8, 8), (6, 10)))


def test_full_size_properties(dct, oracle):
    """BASELINE sizes through size-independent properties: stripes == whole image,
    split == fused, a sampled band against the oracle, checksum of checksums."""
    N = 8192
    g = torch.Generator(device="cuda").manual_seed(42)
    img = torch.randint(0, 256, (N, N), device="cuda", generator=g, dtype=torch.int32).float()
    out = dct.roundtrip(img)
    coef = dct.forward(img)
    rec = dct.inverse(coef)
    assert torch.equal(out.view(torch.int32), rec.view(torch.int32))
    tma, direct = dct.Plan(path=2), dct.Plan(path=1)
    assert torch.equal(dct.roundtrip(img, plan=tma).view(torch.int32), dct.roundtrip(img, plan=direct).view(torch.int32))
    # stripes of block-rows (the multi-GPU partition) reproduce the full result
    for r0, r1 in ((0, 1024), (1024, 1032), (4096, 8192)):
        part = dct.roundtrip(img[r0:r1])
        assert torch.equal(part.view(torch.int32), out[r0:r1].view(torch.int32))
    # bands against the oracle
    for r0 in (0, 4096 + 8, N - 16):
        band = host(img[r0:r0 + 16])
        assert np.array_equal(bits(host(out[r0:r0 + 16])), bits(oracle.roundtrip(band)))
    # u8 at full size: u8 path == f32 path + convertToUnsignedChar
    img8 = img.to(torch.uint8)
    out8 = dct.roundtrip(img8)
    assert torch.equal(out8, out.clamp(0, 255).to(torch.uint8))
    mse, peen = dct.metrics(img8, out8)
    assert 330 < mse < 360 and 12 < peen < 13     # Appendix B: 344.38 / 12.593 on rand()%256 data


def test_two_gigapixel_image_indexing(dct, oracle):
    """Maximum sizes: 65536 x 32768 u8 = 2^31 pixels (the reference's `int` indexing caps
    W*H below 2^31, utils_kernels.cu:12).  Bands at both ends and across the 2^31-byte
    boundary must match the oracle on both kernel families; f32 46344-row strip likewise."""
    H, W = 65536, 32768
    g = torch.Generator(device="cuda").manual_seed(5)
    img = torch.randint(0, 256, (H, W), device="cuda", generator=g, dtype=torch.uint8)
    for path in (1, 2):
        out = dct.roundtrip(img, plan=dct.Plan(path=path))
        for r0 in (0, H // 2 - 8, H - 16):
            band = host(img[r0:r0 + 16])
            assert np.array_equal(host(out[r0:r0 + 16]), oracle.roundtrip(band)), (path, r0)
        del out
    del img
    torch.cuda.empty_cache()
    H, W = 32768 + 8, 32768     # f32: 4 GiB + a block-row, byte offsets beyond 2^32
    imgf = torch.randint(0, 256, (H, W), device="cuda", generator=g, dtype=torch.int32).float()
    out = dct.roundtrip(imgf)
    for r0 in (0, 32768 - 8, H - 8):
        assert np.array_equal(bits(host(out[r0:r0 + 8])), bits(oracle.roundtrip(host(imgf[r0:r0 + 8])))), r0


def test_file_to_file_flow(dct, oracle, tmp_path):
    """The reference program's whole flow (main_newAppr.cu:26-165): image file in, transformed
    image file out.  PGM is lossless, so the file equals the oracle's u8 reconstruction."""
    img = oracle.rand_image_u8(100, 203, 9)             # ragged: cropped to 96 x 200
    src, dst = str(tmp_path / "in.pgm"), str(tmp_path / "out.pgm")
    dct.imageio.save_gray(src, img)
    mse, peen = dct.imageio.transform_file(src, dst)
    want = oracle.roundtrip(np.ascontiguousarray(img[:96, :200]))
    assert np.array_equal(dct.imageio.load_gray(dst), want)
    wm, wp = oracle.metrics(np.ascontiguousarray(img[:96, :200]), want)
    assert mse == pytest.approx(wm, rel=1e-12) and peen == pytest.approx(wp, rel=1e-12)
    jpg = str(tmp_path / "out.jpg")
    dct.imageio.transform_file(src, jpg)                # quality-100 JPEG, as the reference saves
    assert dct.imageio.load_gray(jpg).shape == (96, 200)


@pytest.mark.parametrize("path", ["tma", "direct"])
def test_in_place_calls(dct, oracle, path):
    """out may alias in: every block (tile) is read completely before it is written."""
    img = oracle.rand_image(128, 256, 17)
    plan = dct.Plan(path=PATHS[path])
    d = dev(img)
    dct.roundtrip(d, out=d, plan=plan)
    assert np.array_equal(bits(host(d)), bits(oracle.roundtrip(img)))
    d = dev(img)
    dct.forward(d, coef=d, plan=plan)
    assert np.array_equal(bits(host(d)), bits(oracle.dct(img)))
    dct.inverse(d, img=d, plan=plan)
    assert np.array_equal(bits(host(d)), bits(oracle.roundtrip(img)))
    u8 = dev(img.astype(np.uint8))
    dct.roundtrip(u8, out=u8, plan=plan)
    assert np.array_equal(host(u8), oracle.roundtrip(img.astype(np.uint8)))


@pytest.mark.parametrize("shape", [(1, 1), (7, 9), (100, 203), (64, 70), (37, 256), (256, 256), (1081, 1923)])
@pytest.mark.parametrize("u8", [False, True])
def test_any_size_round_trip(dct, oracle, shape, u8):
    """b200dct_roundtrip_any: ragged sizes run one pass of the edge-replicating kernel (blocks
    sticking out over the edge are completed by edge replication, only the inside is stored);
    equals the oracle applied to the np.pad(mode='edge') image, cropped."""
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    img = rng.integers(0, 256, shape).astype(np.uint8 if u8 else np.float32)
    H, W = shape
    padded = np.pad(img, ((0, -H % 8), (0, -W % 8)), mode="edge")
    want = oracle.roundtrip(np.ascontiguousarray(padded))[:H, :W]
    got = host(dct.roundtrip_any(dev(img)))
    assert np.array_equal(got, want) if u8 else np.array_equal(bits(got), bits(want))
    # unaligned views of an aligned size take the padded path too and stay exact
    if H % 8 == 0 and W % 8 == 0 and W >= 16:
        big = torch.zeros(H, W + 3, dtype=torch.uint8 if u8 else torch.float32, device="cuda")
        big[:, 1:W + 1] = dev(img)
        got = host(dct.roundtrip_any(big[:, 1:W + 1]))
        assert np.array_equal(got, want) if u8 else np.array_equal(bits(got), bits(want))
    # the destination may be a view inside a larger buffer (sentinels survive) or the image itself
    frame = torch.full((H + 2, W + 5), 77, dtype=torch.uint8 if u8 else torch.float32, device="cuda")
    d = dev(img)
    dct.roundtrip_any(d, out=frame[1:H + 1, 2:W + 2])
    f = host(frame)
    assert np.array_equal(f[1:H + 1, 2:W + 2], want) if u8 else np.array_equal(bits(f[1:H + 1, 2:W + 2]), bits(want))
    f[1:H + 1, 2:W + 2] = 77
    assert (f == 77).all()
    dct.roundtrip_any(d, out=d)
    assert np.array_equal(host(d), want) if u8 else np.array_equal(bits(host(d)), bits(want))
    # plans carry over: retained-coefficient mask and a custom table
    keep = oracle.zigzag_mask(7)
    q = (oracle.jpeg_Q() * 0.5 + 3).astype(np.float32)
    want_p = oracle.roundtrip(np.ascontiguousarray(padded), keep=keep, Q=q)[:H, :W]
    got_p = host(dct.roundtrip_any(dev(img), plan=dct.Plan(keep=keep, Q=q)))
    assert np.array_equal(got_p, want_p) if u8 else np.array_equal(bits(got_p), bits(want_p))


@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("shape", [(8, 8), (256, 256), (72, 1056)])
def test_zigzag_coefficient_stream(dct, oracle, shape, u8):
    """Compact coefficient stream (SURVEY 8f.1): block-major int16 in JPEG zig-zag order, written
    by forward / round trip and read back by inverse; same integers as the coefficient plane."""
    img = oracle.rand_image_u8(*shape, 7) if u8 else oracle.rand_image(*shape, 7)
    want_out, want_coef = oracle.roundtrip(img, want_coef=True)
    want_zz = oracle.zigzag_i16(want_coef)
    d = dev(img)
    zz = dct.forward(d, zigzag=True)
    assert dct.api.last_path() == "direct"
    assert zz.shape == (shape[0] // 8, shape[1] // 8, 64) and zz.dtype == torch.int16
    assert np.array_equal(host(zz), want_zz)
    # the inverse from the stream == the inverse from the plane, bit for bit
    rec = dct.inverse(zz, zigzag=True, img_dtype=d.dtype)
    want_rec = oracle.idct(oracle.unzigzag_i16(want_zz))
    want_rec = oracle.to_u8(want_rec) if u8 else want_rec
    assert np.array_equal(host(rec), want_rec)
    if not u8:
        assert np.array_equal(bits(host(rec)), bits(want_out))
    # fused round trip that also emits the stream; padded block-row pitch keeps its sentinels
    bh, bw = shape[0] // 8, shape[1] // 8
    buf = torch.full((bh, bw + 3, 64), -12345, dtype=torch.int16, device="cuda")
    out = dct.roundtrip(d, coef=buf[:, :bw, :], zigzag=True)
    assert np.array_equal(host(out), want_out)
    got = host(buf)
    assert np.array_equal(got[:, :bw, :], want_zz)
    assert (got[:, bw:, :] == -12345).all()
    # the TMA family does not write this layout: forcing it is an error, never a wrong answer
    with pytest.raises(dct.B200DCTError):
        dct.forward(d, zigzag=True, plan=dct.Plan(path=PATHS["tma"]))


@pytest.mark.parametrize("k", [6, 7, 8, 9, 10])
def test_compiled_retained_coefficient_kernels(dct, oracle, k):
    """k = 6..10 of the default tables run kernels with the mask as a compile-time constant
    (dead forward chains, skipped zero terms in the inverse): same bits as masking after the
    fact, on integer, adversarial (ties, -0 coefficients) and non-integer inputs, f32 and u8."""
    keep = oracle.zigzag_mask(k)
    plan = dct.Plan(keep=keep, path=PATHS["direct"])
    for img in (oracle.rand_image(64, 96, k), inputs.adversarial(32), inputs.float_noise(64, 256),
                inputs.smooth_image(128, 128), -inputs.float_noise(16, 64, 3), np.full((8, 32), 3e5, np.float32)):
        want_out, want_coef = oracle.roundtrip(img, keep=keep, want_coef=True)
        coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
        out = dct.roundtrip(dev(img), coef=coef, plan=plan)
        assert dct.api.last_path() == "direct"
        assert np.array_equal(bits(host(coef)), bits(want_coef))
        assert np.array_equal(bits(host(out)), bits(want_out))
        assert np.array_equal(bits(host(dct.roundtrip(dev(img), plan=plan))), bits(want_out))
    for u8 in (oracle.rand_image_u8(72, 1056, k), inputs.adversarial(32).astype(np.uint8)):
        want_out, want_coef = oracle.roundtrip(u8, keep=keep, want_coef=True)
        c16 = torch.empty(u8.shape, dtype=torch.int16, device="cuda")
        out = dct.roundtrip(dev(u8), coef=c16, plan=plan)
        assert np.array_equal(host(out), want_out) and np.array_equal(host(c16), want_coef.astype(np.int16))
        assert np.array_equal(host(dct.roundtrip(dev(u8))), oracle.roundtrip(u8))  # default plan untouched


def test_full_size_masks_and_streams(dct, oracle):
    """BASELINE sizes (8192^2), size-independent properties of the round-1 additions:
    a retained-coefficient mask is applied AFTER quantisation, so the masked coefficient plane
    is the unmasked one with the dropped positions zeroed, on both kernel families and with the
    mask compiled in (k = 6..10) or as data (k = 5); the zig-zag stream is a permutation of the
    int16 plane; fused round trip == forward + inverse; bands against the oracle."""
    N = 8192
    g = torch.Generator(device="cuda").manual_seed(11)
    img = torch.randint(0, 256, (N, N), device="cuda", generator=g, dtype=torch.int32).float()
    full = dct.forward(img)
    rr, cc = torch.meshgrid(torch.arange(N, device="cuda") % 8, torch.arange(N, device="cuda") % 8, indexing="ij")
    pos = rr * 8 + cc
    for k in (5, 6, 10):
        keep = oracle.zigzag_mask(k)
        kept = ((torch.tensor(keep, dtype=torch.int64, device="cuda") >> pos) & 1).bool()
        want = torch.where(kept, full, torch.zeros_like(full))
        for path in (1, 2):
            plan = dct.Plan(keep=keep, path=path)
            coef = torch.empty_like(img)
            out = dct.roundtrip(img, coef=coef, plan=plan)
            assert torch.equal(coef, want), (k, path)          # values (0 == -0 here: signs are checked on the bands)
            assert torch.equal(out.view(torch.int32), dct.inverse(coef, plan=plan).view(torch.int32)), (k, path)
            for r0 in (0, N - 8):
                w_out, w_coef = oracle.roundtrip(host(img[r0:r0 + 8]), keep=keep, want_coef=True)
                assert np.array_equal(bits(host(out[r0:r0 + 8])), bits(w_out)), (k, path, r0)
                assert np.array_equal(bits(host(coef[r0:r0 + 8])), bits(w_coef)), (k, path, r0)
        del want, kept
    # u8 with compiled masks at full size == f32 result through convertToUnsignedChar
    plan = dct.Plan(keep=oracle.zigzag_mask(10))
    out8 = dct.roundtrip(img.to(torch.uint8), plan=plan)
    assert torch.equal(out8, dct.roundtrip(img, plan=plan).clamp(0, 255).to(torch.uint8))
    # zig-zag stream == permuted int16 plane
    zz = dct.forward(img, zigzag=True)
    c16 = dct.forward(img, coef_dtype=torch.int16)
    blocks = c16.view(N // 8, 8, N // 8, 8).permute(0, 2, 1, 3).reshape(N // 8, N // 8, 64)
    order = torch.tensor(oracle.zigzag_i16(np.arange(64, dtype=np.float32).reshape(8, 8))[0, 0].astype(np.int64), device="cuda")
    assert torch.equal(zz, blocks[:, :, order])
    assert torch.equal(dct.inverse(zz, zigzag=True).view(torch.int32), dct.inverse(full).view(torch.int32))


@pytest.mark.parametrize("dtype", [np.float32, np.uint8])
def test_host_pipeline_overlapping_images(dct, oracle, dtype):
    """b200dct_host_pipeline_*: several images in flight at once (pinned buffers, different
    sizes, chunk boundaries inside and across images), each bit-exact against the oracle; tickets
    complete individually."""
    shapes = [(1024, 2048), (8, 64), (2056, 1024), (512, 4096), (1024, 2048)]
    imgs = [(oracle.rand_image(h, w, 10 + i) if dtype == np.float32 else oracle.rand_image_u8(h, w, 10 + i))
            for i, (h, w) in enumerate(shapes)]
    want = [oracle.roundtrip(x) for x in imgs]
    want = [w if dtype == np.float32 else oracle.to_u8(w) for w in want]
    h_in = [torch.from_numpy(x).pin_memory() for x in imgs]
    h_out = [torch.empty_like(x).pin_memory() for x in h_in]
    with dct.HostPipeline(chunk_bytes=1 << 20, slots=3) as pipe:     # small chunks: many per image
        assert pipe.chunk_bytes == 1 << 20
        tickets = [pipe.submit(a, b) for a, b in zip(h_in, h_out)]
        assert tickets == list(range(len(shapes)))
        pipe.wait(tickets[1])
        assert np.array_equal(h_out[0].numpy(), want[0]) and np.array_equal(h_out[1].numpy(), want[1])
        with pytest.raises(dct.B200DCTError):
            pipe.wait(99)                                            # not submitted yet
        with pytest.raises(dct.B200DCTError):
            pipe.submit(torch.zeros(8, 1 << 20), torch.zeros(8, 1 << 20))   # one block-row exceeds a chunk
        pipe.drain()
        for got, w in zip(h_out, want):
            assert np.array_equal(got.numpy(), w)
        # pageable host memory works too (the copies are then synchronous)
        out = np.empty_like(imgs[2])
        t = pipe.submit(imgs[2], out)
        pipe.wait(t)
        assert np.array_equal(out, want[2])
    # the synchronous one-call form still works and can release its per-thread pipeline
    got = dct.roundtrip_host(imgs[0])
    assert np.array_equal(got, want[0])
    assert dct.lib().b200dct_host_release() == 0
    got = dct.roundtrip_host(imgs[3])
    assert np.array_equal(got, want[3])


@pytest.mark.parametrize("W", [8, 13, 256, 523, 1031])
def test_any_size_u8_every_alignment(dct, oracle, W):
    """The word-packed 8-bit any-size kernel: every combination of source and destination byte
    alignment (0..3), row pitches that change the alignment from row to row, widths that end inside
    a word / inside a block / across several 256-pixel warp spans; frames keep their sentinels."""
    H = 21
    rng = np.random.default_rng(W)
    img = rng.integers(0, 256, (H, W)).astype(np.uint8)
    padded = np.pad(img, ((0, -H % 8), (0, -W % 8)), mode="edge")
    want = oracle.roundtrip(np.ascontiguousarray(padded))[:H, :W]
    for pitch_extra in (0, 1, 2, 7):
        for so in range(4):
            for do in range(4):
                src = torch.full((H + 1, W + 8 + pitch_extra), 9, dtype=torch.uint8, device="cuda")
                dst = torch.full((H + 1, W + 8 + pitch_extra), 77, dtype=torch.uint8, device="cuda")
                src[:H, so:so + W] = dev(img)
                dct.roundtrip_any(src[:H, so:so + W], out=dst[:H, do:do + W])
                got = host(dst)
                assert np.array_equal(got[:H, do:do + W], want), (pitch_extra, so, do)
                got[:H, do:do + W] = 77
                assert (got == 77).all(), ("sentinel", pitch_extra, so, do)
        # in place on an unaligned view
        buf = torch.full((H, W + 5 + pitch_extra), 5, dtype=torch.uint8, device="cuda")
        buf[:, 3:3 + W] = dev(img)
        dct.roundtrip_any(buf[:, 3:3 + W], out=buf[:, 3:3 + W])
        got = host(buf)
        assert np.array_equal(got[:, 3:3 + W], want)
        got[:, 3:3 + W] = 5
        assert (got == 5).all()


@pytest.mark.parametrize("shape", [(8, 32), (256, 256), (72, 1056), (1024, 2048)])
def test_fused_metrics_tma_family(dct, oracle, shape):
    """The TMA family's metrics kernel (two input buffers per warp, error taken from the input tile
    in shared memory, 64-bit fixed-point accumulation): pixels and coefficients bit-exact, MSE/PEEN
    to 1e-6 of the oracle's doubles, non-zero count exact, and -- integer accumulation -- the SAME
    value bit for bit from run to run although tiles are scheduled dynamically."""
    img = inputs.float_noise(*shape, seed=5)
    for keep in (dct.ALL_COEFFS, oracle.zigzag_mask(10)):
        want, wcoef = oracle.roundtrip(img, keep=keep, want_coef=True)
        wm, wp = oracle.metrics(img, want)
        plan = dct.Plan(keep=keep, path=PATHS["tma"])
        seen = set()
        for rep in range(4):
            coef = torch.empty(shape, dtype=torch.float32, device="cuda")
            out, (mse, peen, nnz) = dct.roundtrip_with_metrics(dev(img), coef=coef if rep % 2 else None, plan=plan)
            assert dct.api.last_path() == "tma" and dct.api.last_launch_count() == 1
            assert np.array_equal(bits(host(out)), bits(want))
            if rep % 2:
                assert np.array_equal(bits(host(coef)), bits(wcoef))
            assert mse == pytest.approx(wm, rel=1e-6) and peen == pytest.approx(wp, rel=1e-6)
            assert nnz == int(np.count_nonzero(wcoef))
            seen.add((mse, peen))
        assert len(seen) == 1, "fixed-point accumulation must not depend on the tile schedule"
    # accumulating calls ADD into the caller's accumulators on both families
    x = dev(img)
    both = {}
    for path in ("tma", "direct"):
        _, (m1, p1, n1) = dct.roundtrip_with_metrics(x, plan=dct.Plan(path=PATHS[path]))
        assert m1 == pytest.approx(oracle.metrics(img, oracle.roundtrip(img))[0], rel=1e-6)
        assert dct.api.last_path() == path and dct.api.last_launch_count() == 1   # one launch on both families
        both[path] = (m1, p1, n1)
    # same per-block float sums, same 2^-50 fixed point, integer accumulation: the families agree bit for bit
    assert both["tma"] == both["direct"]
    # and the direct family's integer accumulation does not depend on the CTA schedule either
    seen = {dct.roundtrip_with_metrics(x, plan=dct.Plan(path=PATHS["direct"]))[1] for _ in range(4)}
    assert len(seen) == 1
