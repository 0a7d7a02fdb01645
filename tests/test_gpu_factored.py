"""GPU: the library's DEFAULT behaviour for 8-bit pixel output -- the factored (even/odd
butterfly) inverse of Haweel's T (b200dct_inverse_mode, include/b200dct.h).

Contract checked here (BASELINE.json north_star: "quantized integer coefficients must be
bit-exact, reconstructed pixels within +-1 LSB, MSE and PEEN within 1e-3 relative"):
  * quantised coefficients: BIT-EXACT against the oracle / the compiled reference kernels
    (the forward transform and the quantiser are never factored);
  * u8 pixels: max |diff| <= 1 against convertToUnsignedChar(reference IDCT), and the
    FRACTION of differing pixels is measured and bounded (the float value moves by ~1e-5,
    so only pixels whose value sits within that distance of an integer can flip);
  * MSE / PEEN of the u8 result within 1e-3 relative of the reference's;
  * every kernel family computes the same factored arithmetic: tma == direct == any-size
    == inverse-only == fused-metrics, bit for bit;
  * Plan(inverse=INVERSE_EXACT) restores bit-identical u8 pixels.
All other test modules pin B200DCT_INVERSE=exact (tests/conftest.py) and compare bit for bit.
"""
import numpy as np
import pytest
import torch

import inputs
import refgpu

pytestmark = [pytest.mark.gpu, pytest.mark.factored]

PATHS = {"tma": 2, "direct": 1}
MAX_FLIP_FRACTION = 2e-4   # measured on B200: 2-4e-5 on rand()%256 images (printed by the tests)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def lsb_report(got, want, what):
    d = np.abs(got.astype(np.int16) - want.astype(np.int16))
    frac = float((d != 0).mean())
    print(f"[factored] {what}: max |diff| = {int(d.max())} LSB, differing pixels = {int((d != 0).sum())}/{d.size} ({frac:.2e})")
    return int(d.max()), frac


@pytest.mark.parametrize("path", ["tma", "direct"])
@pytest.mark.parametrize("shape", [(8, 32), (256, 256), (72, 1056), (1024, 1024)])
def test_default_u8_round_trip_is_within_one_lsb(dct, oracle, path, shape):
    img = oracle.rand_image_u8(*shape, 42)
    want_out, want_coef = oracle.roundtrip(img, want_coef=True)
    plan = dct.Plan(path=PATHS[path])                      # default inverse mode (AUTO)
    coef = torch.empty(shape, dtype=torch.float32, device="cuda")
    out = dct.roundtrip(dev(img), coef=coef, plan=plan)
    assert dct.api.last_path() == path
    assert np.array_equal(bits(host(coef)), bits(want_coef))          # coefficients stay bit-exact
    mx, frac = lsb_report(host(out), want_out, f"{path} {shape}")
    assert mx <= 1 and frac <= max(MAX_FLIP_FRACTION, 2.0 / img.size)
    a, b = oracle.metrics(img, host(out)), oracle.metrics(img, want_out)
    assert a[0] == pytest.approx(b[0], rel=1e-3) and a[1] == pytest.approx(b[1], rel=1e-3)
    # the exact mode gives the reference's bytes
    exact = dct.Plan(path=PATHS[path], inverse=dct.api.INVERSE_EXACT)
    assert np.array_equal(host(dct.roundtrip(dev(img), plan=exact)), want_out)


def test_all_kernel_families_compute_the_same_factored_arithmetic(dct, oracle):
    shape = (520, 2048 + 32)
    img = oracle.rand_image_u8(*shape, 3)
    d = dev(img)
    direct = dct.roundtrip(d, plan=dct.Plan(path=1))
    tma = dct.roundtrip(d, plan=dct.Plan(path=2))
    assert torch.equal(direct, tma)
    # inverse-only entry point on the same coefficients (f32 plane, i16 plane, zig-zag stream)
    for path in (1, 2):
        plan = dct.Plan(path=path)
        assert torch.equal(dct.inverse(dct.forward(d, plan=plan), plan=plan, img_dtype=torch.uint8), direct)
        c16 = dct.forward(d, plan=plan, coef_dtype=torch.int16)
        assert torch.equal(dct.inverse(c16, plan=plan, img_dtype=torch.uint8), direct)
    zz = dct.forward(d, zigzag=True)
    assert torch.equal(dct.inverse(zz, img_dtype=torch.uint8, zigzag=True), direct)
    # fused metrics kernel: same pixels, and its sums are exactly the metrics of those pixels
    out, (mse, peen, nnz) = dct.roundtrip_with_metrics(d)
    assert torch.equal(out, direct)
    wm, wp = oracle.metrics(img, host(out))
    assert mse == pytest.approx(wm, rel=1e-12) and peen == pytest.approx(wp, rel=1e-12)
    assert nnz == int(np.count_nonzero(oracle.dct(img)))
    # the any-size kernel on an unaligned view of the same pixels
    frame = torch.zeros(shape[0] + 1, shape[1] + 3, dtype=torch.uint8, device="cuda")
    view = frame[1:, 3:]
    view.copy_(d)
    got = dct.roundtrip_any(view)
    assert dct.api.last_path() == "any"
    assert torch.equal(got, direct)
    # host-buffer entry point
    assert np.array_equal(dct.roundtrip_host(img), host(direct))


@pytest.mark.parametrize("shape", [(1, 1), (7, 9), (100, 203), (1081, 1923)])
def test_any_size_u8_default_mode(dct, oracle, shape):
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    img = rng.integers(0, 256, shape).astype(np.uint8)
    H, W = shape
    padded = np.pad(img, ((0, (-H) % 8), (0, (-W) % 8)), mode="edge")
    want = oracle.roundtrip(padded)[:H, :W]
    got = host(dct.roundtrip_any(dev(img)))
    mx, frac = lsb_report(got, want, f"any {shape}")
    assert mx <= 1 and frac <= max(MAX_FLIP_FRACTION, 2.0 / img.size)


def test_adversarial_inputs_stay_within_one_lsb(dct, oracle):
    """Flat / saturated / tie-laden blocks reconstruct onto (almost) exact integers, where the
    truncating u8 conversion (utils.cu:21) amplifies any last-bit difference to a whole LSB --
    in the reference's own float result as much as in the factored one.  The bound is still
    1 LSB; on such images callers who need the reference's bytes use INVERSE_EXACT."""
    for img in (inputs.adversarial(32).astype(np.uint8), np.full((64, 64), 100, np.uint8),
                np.full((64, 64), 255, np.uint8), np.zeros((64, 64), np.uint8),
                inputs.smooth_image(128, 128).astype(np.uint8)):
        want, want_coef = oracle.roundtrip(img, want_coef=True)
        coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
        got = host(dct.roundtrip(dev(img), coef=coef))
        assert np.array_equal(bits(host(coef)), bits(want_coef))
        mx, _ = lsb_report(got, want, f"adversarial {img.shape} mean={img.mean():.1f}")
        assert mx <= 1


def test_custom_tables_and_masks(dct, oracle):
    img = oracle.rand_image_u8(64, 512, 11)
    for Q, keep in ((oracle.jpeg_Q() * 0.5, dct.ALL_COEFFS), (oracle.jpeg_Q(), dct.zigzag_mask(21)),
                    (np.full(64, 1.5, np.float32), dct.ALL_COEFFS), (oracle.jpeg_Q(), dct.zigzag_mask(10))):
        plan = dct.Plan(Q=Q, keep=keep)
        want, want_coef = oracle.roundtrip(img, Q=Q, keep=keep, want_coef=True)
        coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
        got = host(dct.roundtrip(dev(img), coef=coef, plan=plan))
        assert np.array_equal(bits(host(coef)), bits(want_coef))
        mx, frac = lsb_report(got, want, f"Q[0]={Q[0]} keep={keep:#x}")
        assert mx <= 1 and frac <= 1e-3


@pytest.mark.parametrize("N", [2048, 8192])
def test_default_u8_against_the_compiled_reference(dct, oracle, N):
    """The reference's own flow: f32 image -> dct_all_blocks_cuda -> idct_all_blocks_cuda ->
    convertToUnsignedChar (main_newAppr.cu:99-141), against ONE fused u8 -> u8 pass.  Where
    oracle/_ref is not built, the oracle's digests of that flow (tests/golden/refgpu_digests.json,
    checked against the live reference where it is built) stand in for it: the exact-mode
    output must carry exactly those bytes, and then serves as the reference's u8 image."""
    want = refgpu.stored(f"u8flow{N}")
    img8 = dev(oracle.rand_image_u8(N, N, 42))
    exact = dct.roundtrip(img8, plan=dct.Plan(inverse=dct.api.INVERSE_EXACT))
    assert refgpu.digest(exact) == want["u8"]                # exact mode: the stored u8 flow's bytes
    if refgpu.available("newappr"):
        T = dev(oracle.haweel_T())
        refgpu.set_quant("newappr", oracle.jpeg_Q())
        work = img8.float()
        ref_coef, _ = refgpu.dct("newappr", work, T)
        ref_rec, _ = refgpu.idct("newappr", ref_coef, T)
        ref_u8 = ref_rec.clamp(0, 255).to(torch.uint8)       # clamp then truncate == utils.cu:21
        assert refgpu.digest(ref_coef.to(torch.int16)) == want["coef_i16"] and refgpu.digest(ref_u8) == want["u8"]
        del work, ref_coef, ref_rec
    else:
        ref_u8 = exact
    c16 = torch.empty(N, N, dtype=torch.int16, device="cuda")
    out = dct.roundtrip(img8, coef=c16)
    assert refgpu.digest(c16) == want["coef_i16"]            # same integers (int16 carries no sign of zero)
    d = (out.short() - ref_u8.short()).abs()
    n_diff, mx = int((d != 0).sum()), int(d.max())
    print(f"[factored] {N}^2 vs compiled reference: max |diff| = {mx} LSB, differing pixels = {n_diff}/{N * N} ({n_diff / (N * N):.2e})")
    assert mx <= 1 and n_diff <= MAX_FLIP_FRACTION * N * N
    a, b = dct.metrics(img8, out), dct.metrics(img8, ref_u8)
    print(f"[factored] {N}^2 MSE {a[0]:.6f} vs reference {b[0]:.6f}; PEEN {a[1]:.6f} vs {b[1]:.6f}")
    assert b[0] == pytest.approx(want["mse"], rel=1e-12) and b[1] == pytest.approx(want["peen"], rel=1e-12)
    assert a[0] == pytest.approx(b[0], rel=1e-3) and a[1] == pytest.approx(b[1], rel=1e-3)
    # exact mode: the reference's bytes
    assert torch.equal(dct.roundtrip(img8, plan=dct.Plan(inverse=dct.api.INVERSE_EXACT)), ref_u8)


# ------------------------------------------------------------------ dense T with DCT-II symmetry
def test_symmetric_dense_kernels_against_the_chain_oracle(dct, oracle):
    """Default dense mode: a T with symmetric even / antisymmetric odd rows (the true DCT-II) is
    evaluated through its even/odd halves.  Against the ordered-chain oracle: quantised
    coefficients differ by at most 1 and only at (near-)ties -- the same order of magnitude as
    live cuBLAS itself differs from the chain (tests/test_gpu_reference.py); the inverse on
    IDENTICAL coefficients agrees to float re-association noise; both kernel families agree bit
    for bit; a T without the structure, or DENSE_CHAIN, runs the chains == the oracle."""
    T = oracle.dct2_T()
    shape = (520, 2048 + 32)
    img = oracle.rand_image(*shape, 9)
    want_coef = oracle.dct(img, T=T)
    plan = dct.Plan(T=T)
    assert plan.kernel_kind == 2 and not plan.is_sparse
    d = dev(img)
    coef = dct.forward(d, plan=plan)
    diff = (host(coef) - want_coef)
    n_diff = int(np.count_nonzero(diff))
    print(f"[symmetric dense] coefficient mismatches vs ordered-chain oracle: {n_diff}/{img.size} ({n_diff / img.size:.2e}), max |diff| {np.abs(diff).max()}")
    assert np.abs(diff).max() <= 1 and n_diff <= 2e-3 * img.size
    rec = host(dct.inverse(dev(want_coef), plan=plan))
    want_rec = oracle.idct(want_coef, T=T)
    print(f"[symmetric dense] max pixel |diff| on identical coefficients: {np.abs(rec - want_rec).max():.3e}")
    assert np.abs(rec - want_rec).max() < 1e-3
    rec8 = host(dct.inverse(dev(want_coef), plan=plan, img_dtype=torch.uint8))
    mx, frac = lsb_report(rec8, oracle.to_u8(want_rec), "symmetric dense u8")
    assert mx <= 1 and frac <= MAX_FLIP_FRACTION
    # every family / entry point computes the same thing
    c1 = torch.empty_like(d)
    o1 = dct.roundtrip(d, coef=c1, plan=dct.Plan(T=T, path=1))
    c2 = torch.empty_like(d)
    o2 = dct.roundtrip(d, coef=c2, plan=dct.Plan(T=T, path=2))
    assert torch.equal(c1.view(torch.int32), c2.view(torch.int32)) and torch.equal(o1.view(torch.int32), o2.view(torch.int32))
    assert torch.equal(c1.view(torch.int32), coef.view(torch.int32))
    assert torch.equal(dct.inverse(coef, plan=plan).view(torch.int32), o1.view(torch.int32))
    view = torch.zeros(shape[0] + 1, shape[1] + 3, device="cuda")[1:, 3:]
    view.copy_(d)
    assert torch.equal(dct.roundtrip_any(view, plan=plan).view(torch.int32), o1.view(torch.int32))
    # metrics kernel: same pixels
    om, _ = dct.roundtrip_with_metrics(d, plan=plan)
    assert torch.equal(om.view(torch.int32), o1.view(torch.int32))
    # ordered chains on request, and for a T without the symmetry
    chain = dct.Plan(T=T, dense=dct.api.DENSE_CHAIN)
    assert chain.kernel_kind == 0
    assert np.array_equal(bits(host(dct.forward(d, plan=chain))), bits(want_coef))
    assert np.array_equal(bits(host(dct.roundtrip(d, plan=chain))), bits(oracle.roundtrip(img, T=T)))
    T3 = T.copy()
    T3[3 * 8 + 2] *= 1.0009765625
    odd = dct.Plan(T=T3)
    assert odd.kernel_kind == 0
    assert np.array_equal(bits(host(dct.roundtrip(d, plan=odd))), bits(oracle.roundtrip(img, T=T3)))


def test_symmetric_dense_full_size_16384(dct, oracle):
    """BASELINE configs[3]: exact DCT on 16384 x 16384, checked by bands against the oracle
    (mismatch count on the coefficients, float noise on the inverse) and family == family."""
    N = 16384
    T = oracle.dct2_T()
    g = torch.Generator(device="cuda").manual_seed(16384)
    img = torch.randint(0, 256, (N, N), device="cuda", generator=g, dtype=torch.int32).float()
    plan = dct.Plan(T=T)
    coef = dct.forward(img, plan=plan)
    out = dct.roundtrip(img, plan=plan)
    assert torch.equal(dct.inverse(coef, plan=plan).view(torch.int32), out.view(torch.int32))
    tot, bad = 0, 0
    for r0 in (0, 8192 - 8, N - 16):
        band = host(img[r0:r0 + 16])
        wc = oracle.dct(band, T=T)
        dd = host(coef[r0:r0 + 16]) - wc
        assert np.abs(dd).max() <= 1
        bad += int(np.count_nonzero(dd))
        tot += dd.size
        rec = host(dct.inverse(dev(wc), plan=plan))
        assert np.abs(rec - oracle.idct(wc, T=T)).max() < 1e-3
    print(f"[symmetric dense 16384^2] coefficient mismatches vs ordered-chain oracle in 3 bands: {bad}/{tot} ({bad / tot:.2e})")
    assert bad <= 2e-3 * tot
    del coef
    o2 = dct.roundtrip(img, plan=dct.Plan(T=T, path=2))
    assert torch.equal(o2.view(torch.int32), out.view(torch.int32))
    # chain mode at full size == oracle bands, bit for bit
    oc = dct.roundtrip(img, plan=dct.Plan(T=T, dense=dct.api.DENSE_CHAIN))
    for r0 in (0, N - 16):
        assert np.array_equal(bits(host(oc[r0:r0 + 16])), bits(oracle.roundtrip(host(img[r0:r0 + 16]), T=T)))


@pytest.mark.factored
@pytest.mark.parametrize("shape", [(8, 8), (256, 256), (72, 1048), (1024, 1024)])
def test_tensor_core_arm_of_the_dense_variant(dct, oracle, shape):
    """DENSE_MMA (BASELINE configs[3], tensor-core path): batched 8x8 contractions on mma.sync TF32
    with hi/lo operand splits.  Same criterion as every dense-T arithmetic that re-associates sums
    (cuBLAS included): quantised coefficients differ from the ordered FP32 chain in at most a few
    1e-4 of the positions and then by one step; pixels within 1 LSB after the 8-bit conversion;
    MSE / PEEN within 1e-3."""
    T = oracle.dct2_T()
    img = oracle.rand_image(*shape, 11)
    want, wcoef = oracle.roundtrip(img, T=T, want_coef=True)
    plan = dct.Plan(T=T, dense=dct.api.DENSE_MMA)
    d = torch.from_numpy(img).cuda()
    coef = torch.empty_like(d)
    out = dct.roundtrip(d, coef=coef, plan=plan)
    assert dct.api.last_path() == "mma"
    torch.cuda.synchronize()
    gc, go = coef.cpu().numpy(), out.cpu().numpy()
    diff = np.abs(gc - wcoef)
    frac = float(np.mean(diff > 0))
    assert diff.max() <= 1 and frac < 2e-3, (diff.max(), frac)
    same = diff.reshape(shape[0] // 8, 8, shape[1] // 8, 8).max(axis=(1, 3)) == 0       # blocks with identical coefficients
    pix = np.abs(go - want).reshape(shape[0] // 8, 8, shape[1] // 8, 8).max(axis=(1, 3))
    assert pix[same].max() < 2e-3                                                        # same coefficients -> same pixels up to FP32 rounding
    assert np.abs(oracle.to_u8(go).astype(np.int16) - oracle.to_u8(want).astype(np.int16)).max() <= 1 or frac > 0
    m_w, p_w = oracle.metrics(img, want)
    m_g, p_g = oracle.metrics(img, go)
    assert abs(m_g - m_w) <= 1e-3 * m_w and abs(p_g - p_w) <= 1e-3 * p_w
    # without the coefficient plane, masks and custom tables, non-integer divisors (IEEE division kernel)
    out2 = dct.roundtrip(d, plan=plan)
    assert torch.equal(out2, out)
    for Q, keep in ((oracle.jpeg_Q() * 2, oracle.zigzag_mask(10)), (oracle.jpeg_Q() * 0.37, dct.ALL_COEFFS)):
        w2, c2 = oracle.roundtrip(img, T=T, Q=Q, keep=keep, want_coef=True)
        cf = torch.empty_like(d)
        dct.roundtrip(d, coef=cf, plan=dct.Plan(T=T, Q=Q, keep=keep, dense=dct.api.DENSE_MMA))
        dd = np.abs(cf.cpu().numpy() - c2)
        assert dd.max() <= 1 and np.mean(dd > 0) < 2e-3
    # every other call of such a plan runs the CUDA-core kernels
    c16 = dct.forward(d, plan=plan)
    assert dct.api.last_path() in ("direct", "tma")
