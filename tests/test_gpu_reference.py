"""GPU: the UNMODIFIED reference kernels (oracle/_ref, compiled from the reference's sources by
oracle/Makefile) against (a) the CPU oracle -- this is what pins the oracle -- and
(b) the new CUDA path.  Bit-exact for HpApprDCT and fastApprDCT.  (b) also runs where
oracle/_ref is not built: it then compares against tests/golden/refgpu_digests.json, digests of
the CPU oracle's outputs for the same inputs.  The oracle reproduces the reference bit for bit
on the reference outputs committed as tests/golden/refgpu_*.npz and on SURVEY.md Appendix B,
and wherever oracle/_ref is built these tests check every digest they use against the live
reference too.  Without it, (a) only checks that the oracle still produces its stored digests:
a regression guard, not a comparison with the reference; and the fastappr cases repeat the
newappr ones, as both reference programs compute the same bits.  The two cuBLAS variants accumulate in an order cuBLAS does not document, so for them the
mismatch COUNT is reported and bounded (SURVEY.md section 7.3 item 3), pixels within +-1 LSB;
they need the live reference."""
import os

import numpy as np
import pytest
import torch

import inputs
import refgpu

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def need(variant):
    if not refgpu.available(variant):
        pytest.skip(f"oracle/_ref/{refgpu.VARIANTS[variant]} not built (needs the reference's sources at build time)")


def live_reference(o, variant, img, Q=None):
    """(coef, image left behind, rec) of the live reference kernels as host arrays, or None
    where oracle/_ref is not built."""
    if not refgpu.available(variant):
        return None
    T = dev(o.haweel_T())
    rc = refgpu.set_quant(variant, o.jpeg_Q() if Q is None else Q)
    if Q is not None:
        assert rc == 0          # a custom Q must reach the reference (fastApprDCT hard-codes JPEG Q and reports -1)
    d_img = dev(img)
    ref_coef, _ = refgpu.dct(variant, d_img, T)
    ref_rec, _ = refgpu.idct(variant, ref_coef, T)
    res = host(ref_coef), host(d_img), host(ref_rec)
    refgpu.set_quant(variant, o.jpeg_Q())
    return res


def check_stored(case, coef=None, shifted=None, rec=None):
    """The given arrays carry the stored bits for `case` (tests/golden/refgpu_digests.json: the
    oracle's outputs, equal to the reference's wherever the two have been compared)."""
    want = refgpu.stored(case)
    for name, a in (("coef", coef), ("shifted", shifted), ("rec", rec)):
        if a is not None:
            assert refgpu.digest(a) == want[name], f"{case}: {name} differs from the stored oracle digest"


@pytest.mark.parametrize("variant", ["newappr", "fastappr"])
@pytest.mark.parametrize("N", [256, 512, 1024, 2048])
def test_reference_kernels_pin_the_oracle(oracle, dct, variant, N):
    case = f"rand{N}"
    img = oracle.rand_image(N, N, 42)
    want_coef, want_shift = oracle.dct(img, want_shifted=True)
    want_rec = oracle.idct(want_coef)
    ref = live_reference(oracle, variant, img)
    if ref is not None:
        # (a) oracle == live reference, bit for bit (including the sign of zero coefficients)
        assert np.array_equal(bits(ref[0]), bits(want_coef))
        assert np.array_equal(ref[1], want_shift)                     # input left as image-128
        assert np.array_equal(bits(ref[2]), bits(want_rec))
        check_stored(case, *ref)                                      # the stored digests are the reference's
    # the oracle still produces its stored digests (without oracle/_ref: a regression guard only)
    check_stored(case, want_coef, want_shift, want_rec)
    # (b) new CUDA path == reference (live above, or through the oracle's stored digests)
    d2 = dev(img)
    coef = torch.empty_like(d2)
    out = dct.roundtrip(d2, coef=coef)
    check_stored(case, coef=coef, rec=out)
    # MSE / PEEN of the u8 result agree (spec: 1e-3 relative)
    u8 = d2.to(torch.uint8)
    m_new = dct.metrics(u8, out.clamp(0, 255).to(torch.uint8))
    m_ref = refgpu.stored(case)["mse"], refgpu.stored(case)["peen"]
    if ref is not None:
        live = dct.metrics(u8, dev(ref[2]).clamp(0, 255).to(torch.uint8))
        assert live[0] == pytest.approx(m_ref[0], rel=1e-12) and live[1] == pytest.approx(m_ref[1], rel=1e-12)
    assert m_new[0] == pytest.approx(m_ref[0], rel=1e-12) and m_new[1] == pytest.approx(m_ref[1], rel=1e-12)


def test_headline_size_whole_image_against_the_reference_kernel(oracle, dct):
    """BASELINE configs[1] compared WHOLE: every coefficient and every f32 pixel of the 8192^2
    image against the unmodified reference kernels (3.3 ms on a B200) or, without them, the
    oracle's stored digests, plus SURVEY.md Appendix B's N=8192 known answers on the GPU results."""
    N = 8192
    img = oracle.rand_image(N, N, 42)                       # srand(42); rand()%256
    ref = live_reference(oracle, "newappr", img)
    if ref is not None:
        check_stored("rand8192", coef=ref[0], rec=ref[2])
        del ref
    d = dev(img)
    for path in (2, 1):
        plan = dct.Plan(path=path)
        coef = torch.empty_like(d)
        out = dct.roundtrip(d, coef=coef, plan=plan)
        check_stored("rand8192", coef=coef, rec=out)
    # the split entry points (the drop-in two-call API) as well
    c2 = dct.forward(d)
    check_stored("rand8192", coef=c2, rec=dct.inverse(c2))
    # Appendix B, N = 8192
    assert int(coef.double().sum().item()) == -268447
    assert int(coef.abs().double().sum().item()) == 117045095
    assert int((coef != 0).sum().item()) == 47462419
    u8 = out.clamp(0, 255).to(torch.uint8)
    assert int(u8.long().sum().item()) == 8524699637
    mse, peen = dct.metrics(d.to(torch.uint8), u8)
    assert mse == pytest.approx(344.379744306, rel=1e-9) and peen == pytest.approx(12.593068395, rel=1e-9)


def test_reference_on_adversarial_and_rectangular(oracle, dct):
    for case, img in (("adversarial32", inputs.adversarial(32)), ("floatnoise64x256", inputs.float_noise(64, 256)),
                      ("rand48x640_seed7", oracle.rand_image(48, 640, 7))):
        ref = live_reference(oracle, "newappr", img)
        if ref is not None:
            assert np.array_equal(bits(ref[0]), bits(oracle.dct(img)))
            assert np.array_equal(bits(ref[2]), bits(oracle.idct(oracle.dct(img))))
            check_stored(case, coef=ref[0], rec=ref[2])
        check_stored(case, coef=oracle.dct(img), rec=oracle.idct(oracle.dct(img)))
        check_stored(case, rec=dct.roundtrip(dev(img)))


def test_reference_custom_quant(oracle, dct):
    img = oracle.rand_image(256, 256, 5)
    Q = oracle.jpeg_Q() * 0.5
    ref = live_reference(oracle, "newappr", img, Q=Q)
    if ref is not None:
        assert np.array_equal(bits(ref[0]), bits(oracle.dct(img, Q=Q)))
        check_stored("rand256_seed5_halfq", coef=ref[0])
    check_stored("rand256_seed5_halfq", coef=oracle.dct(img, Q=Q))
    check_stored("rand256_seed5_halfq", coef=dct.forward(dev(img), plan=dct.Plan(Q=Q)))


@pytest.mark.parametrize("variant", ["cublas2", "cublas"])
def test_cublas_variants_mismatch_count(oracle, dct, variant):
    """cuBLAS's k-accumulation order is opaque: report how many coefficients differ from
    the FMA-chain result, require pixels within +-1 LSB and MSE/PEEN within 1e-3."""
    need(variant)
    N = 256
    img = oracle.rand_image(N, N, 42)
    refgpu.set_quant(variant, oracle.jpeg_Q())
    for name, Tm in (("haweel", oracle.haweel_T()), ("dct2", oracle.dct2_T())):
        T = dev(Tm)
        d_img = dev(img)
        ref_coef, _ = refgpu.dct(variant, d_img, T)
        keep = ref_coef.clone()
        ref_rec, _ = refgpu.idct(variant, ref_coef, T)     # v2 dequantises ref_coef in place
        plan = dct.Plan(T=Tm)
        coef = dct.forward(dev(img), plan=plan)
        rec = dct.inverse(keep, plan=plan)                  # same coefficients in: isolates the inverse
        n_diff = int((coef != keep).sum())
        max_cdiff = float((coef - keep).abs().max())
        pix_diff = float((rec - ref_rec).abs().max())
        print(f"[{variant}/{name}] coefficient mismatches vs cuBLAS: {n_diff}/{N * N} (max |diff| {max_cdiff}); "
              f"max pixel diff for identical coefficients: {pix_diff:.3e}")
        assert max_cdiff <= 1 and n_diff <= N * N * 2e-3
        assert pix_diff < 1e-3                               # float reassociation noise only
        u8 = dev(img).to(torch.uint8)
        a = dct.metrics(u8, rec.clamp(0, 255).to(torch.uint8))
        b = dct.metrics(u8, ref_rec.clamp(0, 255).to(torch.uint8))
        assert a[0] == pytest.approx(b[0], rel=1e-3) and a[1] == pytest.approx(b[1], rel=1e-3)
        assert int((rec.clamp(0, 255).to(torch.uint8).int() - ref_rec.clamp(0, 255).to(torch.uint8).int()).abs().max()) <= 1


@pytest.mark.factored
@pytest.mark.parametrize("N", [1024, 2048])
def test_cublas2_mismatch_counts_at_larger_sizes(oracle, dct, N):
    """cublasDCTv2 (whole-image Sgemm, main_cublass_2.cu:228-235,288-295) at 1024^2 and 2048^2 with
    the true DCT-II matrix: mismatch count of the quantised coefficients for BOTH dense modes
    (ordered chains, and the default even/odd evaluation) -- the even/odd kernel must be no
    further from cuBLAS than the chain kernel is, pixels within 1 LSB, MSE/PEEN within 1e-3."""
    need("cublas2")
    img = oracle.rand_image(N, N, 42)
    Tm = oracle.dct2_T()
    refgpu.set_quant("cublas2", oracle.jpeg_Q())
    T = dev(Tm)
    ref_coef, _ = refgpu.dct("cublas2", dev(img), T)
    keep = ref_coef.clone()
    ref_rec, _ = refgpu.idct("cublas2", ref_coef, T)       # dequantises ref_coef in place
    counts = {}
    for name, mode in (("chain", dct.api.DENSE_CHAIN), ("symmetric", dct.api.DENSE_AUTO)):
        plan = dct.Plan(T=Tm, dense=mode)
        coef = dct.forward(dev(img), plan=plan)
        counts[name] = int((coef != keep).sum())
        assert float((coef - keep).abs().max()) <= 1
        rec = dct.inverse(keep, plan=plan)
        assert float((rec - ref_rec).abs().max()) < 1e-3
        u8 = dev(img).to(torch.uint8)
        a = dct.metrics(u8, rec.clamp(0, 255).to(torch.uint8))
        b = dct.metrics(u8, ref_rec.clamp(0, 255).to(torch.uint8))
        assert a[0] == pytest.approx(b[0], rel=1e-3) and a[1] == pytest.approx(b[1], rel=1e-3)
        assert int((rec.clamp(0, 255).to(torch.uint8).int() - ref_rec.clamp(0, 255).to(torch.uint8).int()).abs().max()) <= 1
    # the tensor-core arm (fused round trip only): same criterion against the live cuBLAS result
    cm = torch.empty(N, N, device="cuda")
    om = dct.roundtrip(dev(img), coef=cm, plan=dct.Plan(T=Tm, dense=dct.api.DENSE_MMA))
    assert dct.api.last_path() == "mma"
    counts["mma"] = int((cm != keep).sum())
    assert float((cm - keep).abs().max()) <= 1
    u8 = dev(img).to(torch.uint8)
    a = dct.metrics(u8, om.clamp(0, 255).to(torch.uint8))
    b = dct.metrics(u8, ref_rec.clamp(0, 255).to(torch.uint8))
    assert a[0] == pytest.approx(b[0], rel=1e-3) and a[1] == pytest.approx(b[1], rel=1e-3)
    same = (cm == keep).view(N // 8, 8, N // 8, 8).all(dim=3).all(dim=1)                # blocks with identical coefficients
    pd = (om - ref_rec).abs().view(N // 8, 8, N // 8, 8).amax(dim=3).amax(dim=1)
    assert float(pd[same].max()) < 2e-3
    print(f"[cublas2/dct2 {N}^2] coefficient mismatches vs live cuBLAS: chain {counts['chain']}, "
          f"even/odd {counts['symmetric']}, tensor-core arm {counts['mma']} of {N * N}")
    assert counts["symmetric"] <= max(2 * counts["chain"], 1e-3 * N * N)
    assert counts["mma"] <= 2e-3 * N * N


def test_committed_reference_fixtures_match_live_reference(oracle, dct):
    """tests/golden/refgpu_*.npz were produced by these same reference kernels (checked where
    oracle/_ref is built); the new CUDA path reproduces their coefficients and pixels."""
    import glob

    files = sorted(glob.glob(os.path.join(GOLD, "refgpu_*.npz")))
    assert files, "tests/golden/refgpu_*.npz missing"
    for f in files:
        g = np.load(f)
        img = g["img"].astype(np.float32)
        if refgpu.available("newappr"):
            T = dev(oracle.haweel_T())
            refgpu.set_quant("newappr", oracle.jpeg_Q())
            coef, _ = refgpu.dct("newappr", dev(img), T)
            assert np.array_equal(bits(host(coef)), bits(g["coef"]))
        coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
        out = dct.roundtrip(dev(img), coef=coef)
        assert np.array_equal(bits(host(coef)), bits(g["coef"])), f
        assert np.array_equal(bits(host(out)), bits(g["rec"])), f


def test_cpp_caller_links_against_compat_library(oracle, dct):
    """tests/cpp/dropin_main.cu is written like the reference's programs (forward-declared
    dct_all_blocks_cuda / idct_all_blocks_cuda, (height, width) order, device buffers) and is
    linked against libb200dct_compat.so: it must print the oracle's (= the reference's) numbers."""
    import re
    import subprocess

    exe = os.path.join(os.path.dirname(GOLD.rstrip("/")), "..", "cuda-dct-idct_b200", "dropin_demo")
    exe = os.path.abspath(exe)
    if not os.path.exists(exe):
        pytest.skip("dropin_demo not built")
    for variant in (0, 1):
        out = subprocess.run([exe, "256", str(variant)], capture_output=True, text=True, timeout=120).stdout
        m = re.search(r"COEF sum=(-?\d+) sumabs=(\d+) nonzero=(\d+)", out)
        assert m, out
        assert tuple(map(int, m.groups())) == (-306, 114414, 46317)         # SURVEY.md Appendix B, N=256
        assert int(re.search(r"PIX sumu8=(\d+)", out).group(1)) == 8329775
        assert "DCT (256,256):" in out and "IDCT (256,256):" in out          # the reference's timing lines
        assert "INPUT_AFTER first=-58 (was 70)" in out                       # input left as image-128
