"""GPU: the kernels that re-associate their f32 sums, against the float64 reference of tests/f64ref.py.

Criterion (derived in f64ref.py, no statistical allowance): a quantised coefficient equals
round_half_away(Y/Q) of the exact Y unless Y/Q lies within the rounding bound of a half-integer, and
then it is one of the two neighbours; f32 pixels lie within the bound of the exact pixels of the
kernel's OWN coefficients; u8 pixels equal clamp-then-truncate of those, except where an integer lies
within the bound.  Every plan sets its mode explicitly (DENSE_SYMMETRIC, INVERSE_FACTORED, DENSE_MMA),
so nothing here depends on the environment pin of tests/conftest.py.  Each case prints its largest
error in units of u*B (for u8 outputs and quantised coefficients: the smallest error that explains a
flip) and its ambiguous fraction; the module prints the maximum per arithmetic at the end.

Kernel instances reached (qm: y1/s1 = runtime table, fast division; y2/s2 = IEEE division; s0 = the
JPEG table as immediates):
  symmetric dense T (forward_block_sym / inverse_block_sym), kernel_kind 2:
    k_direct y1/y2 RT, FWD, INV x f32/u8    test_symmetric_dense[direct-*], test_symmetric_shapes, test_symmetric_scale_sweep
    k_direct y1/y2 metrics x f32/u8        test_symmetric_families
    k_tma y1/y2 RT, FWD, INV x f32/u8       test_symmetric_dense[tma-*], test_symmetric_shapes
    k_any y1/y2 TK_DENSE_SYM f32/u8         test_symmetric_families (unaligned view)
    batch (k_direct y1/y2 RT)              test_symmetric_families
  factored inverse of Haweel's T (inverse_block_fast, u8 output):
    k_direct s0/s1/s2 FINV RT, INV u8       test_factored_inverse[direct-*], test_factored_shapes
    k_direct s0/s1/s2 FINV metrics          test_factored_families
    k_tma s0/s1/s2 FINV RT, INV u8          test_factored_inverse[tma-*], test_factored_shapes
    k_any_u8 s0/s1/s2 FINV, batch, host pipeline (roundtrip_host, HostPipeline)   test_factored_families
    k_rgb<qk, FINV, zz> / k_rgb_inverse<FINV>   test_colour (qk 0, 1, 2; with and without streams)
  tensor-core arm: k_mma<true>, k_mma<false>    test_tensor_core_arm, test_tensor_core_scale_sweep
The TMA family has no zig-zag planes (b200dct.cu tma_plane_ok), so zig-zag streams run on the direct
family only.  k_tma has no metrics instance for these arithmetics: the fused metrics of a dense or u8
round trip always run on the direct family (b200dct.cu metrics_tma_ok).
"""
from __future__ import annotations

import numpy as np
import pytest

import f64ref as R
import inputs

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

F32 = np.float32
PATHS = {"direct": 1, "tma": 2}
QNAMES = ["jpeg", "jpeg_x2", "jpeg_mask21", "jpeg_x037"]
SCALES = [-12, -6, -1, 0, 3, 8, 12, 16]     # tests/test_gpu_range.py
WORST: dict = {}
# on random pixels the bound must decide almost everywhere (measured on B200: <= 3.7e-3); flat and
# DC-only blocks reconstruct onto near-integers, which no sound bound decides, so other inputs are exempt
MAX_AMBIGUOUS_RANDOM = 1e-2


@pytest.fixture(scope="module", autouse=True)
def _summary():
    yield
    for k, (w, a) in sorted(WORST.items()):
        print(f"[reassoc] max over the module: {k}: worst {w:.2f} uB, ambiguous <= {a:.2e}")


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def same(a, b):
    if a.dtype == torch.float32:
        return torch.equal(a.view(torch.int32), b.view(torch.int32))
    return torch.equal(a, b)


def record(arith, what, ch, random_input=False):
    print(f"[reassoc] {arith} {what}: {ch}")
    w, a = WORST.get(arith, (0.0, 0.0))
    WORST[arith] = (max(w, ch.worst), max(a, ch.ambiguous))
    assert ch.bad == 0, f"{arith} {what}: {ch}"
    assert not random_input or ch.ambiguous <= MAX_AMBIGUOUS_RANDOM, f"{arith} {what}: {ch}"


def q_of(oracle, qname, dct):
    Q = oracle.jpeg_Q()
    if qname == "jpeg_x2":
        return (Q * F32(2)).astype(F32), dct.ALL_COEFFS
    if qname == "jpeg_x037":
        return (Q * F32(0.37)).astype(F32), dct.ALL_COEFFS
    if qname == "jpeg_mask21":
        return Q, dct.zigzag_mask(21)
    return Q, dct.ALL_COEFFS


def T_of(oracle, tname):
    return oracle.dct2_T() if tname == "dct2" else R.rand_sym_T()


def check_coef(arith, what, C, Y, B, Q, keep, c=R.C_F, random_input=False):
    record(arith + " coef", what, R.check_quant(C, Y, B, Q, keep, c), random_input)


def check_pix(arith, what, out, C, T, Q, c=R.C_I, random_input=False):
    P, Bi = R.inverse64(C, T, Q)
    record(arith, what, R.check_u8(out, P, Bi, c) if out.dtype == np.uint8 else R.check_close(out, P, Bi, c), random_input)


def check_forward_exact(arith, what, dct, d, Y, B, T, c, **plan_kw):
    """The kernel's unquantised Y: with Q = 2^-k (IEEE-division kernels) the coefficient is Y 2^k rounded
    to an integer, which is Y 2^k itself for every |Y| above 2^-k (k chosen so that Y 2^k stays < 2^100)."""
    k = 100 - int(np.ceil(np.log2(max(float(B.max()), 1e-30))))
    plan = dct.Plan(T=T, Q=np.full(64, 2.0 ** -k, F32), **plan_kw)
    coef = torch.empty(d.shape, dtype=torch.float32, device="cuda")
    if plan_kw.get("dense") == dct.api.DENSE_MMA:
        dct.roundtrip(d, coef=coef, plan=plan)
        assert dct.api.last_path() == "mma"
    else:
        dct.forward(d, coef, plan=plan)
    record(arith + " forward", what, R.check_close(host(coef).astype(np.float64) * 2.0 ** -k, Y, B, c))


def u8_image(H, W, seed):
    return inputs.splitmix_u8(H * W, seed).reshape(H, W)


# ---------------------------------------------------------------- symmetric dense T
def run_symmetric(dct, oracle, arith, img, T, Q, keep, path, what, random_input=False):
    """Every entry point of one plan on one image: round trip with each coefficient plane, forward to each
    plane, inverse from each plane to both pixel types."""
    plan = dct.Plan(T=T, Q=Q, keep=keep, path=PATHS[path], dense=dct.api.DENSE_SYMMETRIC)
    assert plan.kernel_kind == 2 and not plan.is_sparse
    d = dev(img)
    Y, B = R.forward64(img, T)
    coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
    out = dct.roundtrip(d, coef=coef, plan=plan)
    assert dct.api.last_path() == path
    C = host(coef)
    check_coef(arith, what, C, Y, B, Q, keep, random_input=random_input)
    check_pix(arith, what + " rt", host(out), C, T, Q, random_input=random_input)
    # the other coefficient planes: same pixels, and the integers of the f32 plane bit for bit
    assert same(dct.roundtrip(d, plan=plan), out)
    c16 = torch.empty(img.shape, dtype=torch.int16, device="cuda")
    assert same(dct.roundtrip(d, coef=c16, plan=plan), out)
    assert np.array_equal(host(c16), C.astype(np.int16))
    zz = None
    if path == "direct":
        zz = dct.api.empty_zigzag(*img.shape, "cuda")
        assert same(dct.roundtrip(d, coef=zz, plan=plan, zigzag=True), out)
        assert np.array_equal(R.unzigzag(host(zz)), C)
    # forward to each plane
    assert same(dct.forward(d, plan=plan), coef)
    assert dct.api.last_path() == path
    assert np.array_equal(host(dct.forward(d, plan=plan, coef_dtype=torch.int16)), C.astype(np.int16))
    if zz is not None:
        assert torch.equal(dct.forward(d, plan=plan, zigzag=True), zz)
    # inverse from each plane to both pixel types
    for odt in (torch.float32, torch.uint8):
        for src, zig in ((coef, False), (c16, False), (zz, True)):
            if src is None:
                continue
            got = dct.inverse(src, plan=plan, img_dtype=odt, zigzag=zig)
            assert dct.api.last_path() == path
            check_pix(arith, f"{what} inv {src.dtype}{' zz' if zig else ''}->{odt}", host(got), C, T, Q,
                      random_input=random_input)
    return plan, C


@pytest.mark.parametrize("pix", ["f32", "u8"])
@pytest.mark.parametrize("path", ["direct", "tma"])
@pytest.mark.parametrize("qname", QNAMES)
@pytest.mark.parametrize("tname", ["dct2", "randsym"])
def test_symmetric_dense(dct, oracle, tname, qname, path, pix):
    T = T_of(oracle, tname)
    Q, keep = q_of(oracle, qname, dct)
    img = u8_image(520, 2080, 7) if pix == "u8" else inputs.float_noise(520, 2080)
    run_symmetric(dct, oracle, "symmetric", img, T, Q, keep, path, f"{tname} {qname} {path} {pix}", random_input=True)
    if qname == "jpeg":
        Y, B = R.forward64(img, T)
        check_forward_exact("symmetric", f"{tname} {path} {pix}", dct, dev(img), Y, B, T, R.C_F,
                            path=PATHS[path], dense=dct.api.DENSE_SYMMETRIC)


# the TMA family needs 16-byte rows (f32: W % 32 == 0), so 8 x 8 runs on the direct family only
SHAPE_PATHS = [((8, 8), "direct"), ((72, 1056), "direct"), ((72, 1056), "tma"), ((2048, 2048), "direct"),
               ((2048, 2048), "tma")]


@pytest.mark.parametrize("shape,path", SHAPE_PATHS)
def test_symmetric_shapes(dct, oracle, shape, path):
    T, Q = oracle.dct2_T(), oracle.jpeg_Q()
    H, W = shape
    adv = np.tile(inputs.adversarial(W // 8), (H // 128 + 1, 1))[:H]
    for name, img in (("rand", u8_image(H, W, 3)), ("adversarial", adv), ("smooth", inputs.smooth_image(H, W)),
                      ("float_noise", inputs.float_noise(H, W, 5))):
        run_symmetric(dct, oracle, "symmetric", img, T, Q, dct.ALL_COEFFS, path, f"{shape} {name} {path}")


@pytest.mark.parametrize("tname", ["dct2", "randsym"])
def test_symmetric_scale_sweep(dct, oracle, tname):
    """y1 and y2 over the scale sweep of test_gpu_range.py: 2^k Q moves between the fast-division and
    the IEEE-division kernels."""
    T = T_of(oracle, tname)
    rng = np.random.default_rng(21)
    x0 = rng.integers(0, 256, (256, 256)).astype(F32)
    x0[:128] = inputs.adversarial(32)
    for k in SCALES:
        s = F32(2.0 ** k)
        x = (F32(128) + s * (x0 - F32(128))).astype(F32)
        Q = (oracle.jpeg_Q() * s).astype(F32)
        plan = dct.Plan(T=T, Q=Q, dense=dct.api.DENSE_SYMMETRIC)
        assert plan.kernel_kind == 2
        d = dev(x)
        coef = torch.empty_like(d)
        out = dct.roundtrip(d, coef=coef, plan=plan)
        Y, B = R.forward64(x, T)
        C = host(coef)
        check_coef("symmetric", f"{tname} scale 2^{k}", C, Y, B, Q, dct.ALL_COEFFS)
        check_pix("symmetric", f"{tname} scale 2^{k}", host(out), C, T, Q)
        check_forward_exact("symmetric", f"{tname} scale 2^{k}", dct, d, Y, B, T, R.C_F, dense=dct.api.DENSE_SYMMETRIC)


@pytest.mark.parametrize("pix", ["f32", "u8"])
@pytest.mark.parametrize("qname", QNAMES)
@pytest.mark.parametrize("tname", ["dct2", "randsym"])
def test_symmetric_families(dct, oracle, tname, qname, pix):
    """Any-size kernel on an unaligned view, batches, and the fused metrics kernel, at a TMA tile edge."""
    T = T_of(oracle, tname)
    Q, keep = q_of(oracle, qname, dct)
    H, W = 72, 1056
    imgs = [u8_image(H, W, s) if pix == "u8" else inputs.float_noise(H, W, s) for s in (1, 2, 3)]
    plan = dct.Plan(T=T, Q=Q, keep=keep, dense=dct.api.DENSE_SYMMETRIC)
    Cs = []
    for img in imgs:
        coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
        dct.forward(dev(img), coef, plan=plan)
        Y, B = R.forward64(img, T)
        Cs.append(host(coef))
        check_coef("symmetric", f"{tname} {qname} families {pix}", Cs[-1], Y, B, Q, keep)
    what = f"{tname} {qname} {pix}"
    outs = dct.roundtrip_batch([dev(i) for i in imgs], plan=plan)
    assert dct.api.last_path() == "direct"
    for o, C in zip(outs, Cs):
        check_pix("symmetric", what + " batch", host(o), C, T, Q)
    d = dev(imgs[0])
    frame = torch.zeros(H + 1, W + 3, dtype=d.dtype, device="cuda")
    view = frame[1:, 3:]
    view.copy_(d)
    got = dct.roundtrip_any(view, plan=plan)
    assert dct.api.last_path() == "any"
    check_pix("symmetric", what + " any", host(got), Cs[0], T, Q)
    out, (mse, peen, nnz) = dct.roundtrip_with_metrics(d, plan=plan)
    assert dct.api.last_path() == "direct"
    o = host(out)
    check_pix("symmetric", what + " metrics", o, Cs[0], T, Q)
    wm, wp = oracle.metrics(imgs[0], o)
    rel = 1e-12 if pix == "u8" else 1e-6
    assert mse == pytest.approx(wm, rel=rel) and peen == pytest.approx(wp, rel=rel)
    assert nnz == int(np.count_nonzero(Cs[0]))


# ---------------------------------------------------------------- factored inverse of Haweel's T (u8)
def factored_plan(dct, Q, keep, path=0):
    plan = dct.Plan(Q=Q, keep=keep, path=path, inverse=dct.api.INVERSE_FACTORED)
    assert plan.kernel_kind == 1 and plan.is_sparse
    return plan


def run_factored(dct, oracle, img, Q, keep, path, what, random_input=False):
    T = oracle.haweel_T()
    plan = factored_plan(dct, Q, keep, PATHS[path])
    d = dev(img)
    coef = torch.empty(img.shape, dtype=torch.float32, device="cuda")
    out = dct.roundtrip(d, coef=coef, plan=plan)
    assert dct.api.last_path() == path
    C = host(coef)
    assert np.array_equal(C.view(np.uint32), oracle.dct(img, Q=Q, keep=keep).view(np.uint32))    # the forward is the chain
    Y, B = R.forward64(img, T)
    check_coef("factored", what, C, Y, B, Q, keep, random_input=random_input)
    check_pix("factored", what + " rt", host(out), C, T, Q, random_input=random_input)
    assert same(dct.roundtrip(d, plan=plan), out)
    c16 = torch.empty(img.shape, dtype=torch.int16, device="cuda")
    assert same(dct.roundtrip(d, coef=c16, plan=plan), out)
    assert np.array_equal(host(c16), C.astype(np.int16))
    zz = None
    if path == "direct":
        zz = dct.api.empty_zigzag(*img.shape, "cuda")
        assert same(dct.roundtrip(d, coef=zz, plan=plan, zigzag=True), out)
        assert np.array_equal(R.unzigzag(host(zz)), C)
    for src, zig in ((coef, False), (c16, False), (zz, True)):
        if src is None:
            continue
        got = dct.inverse(src, plan=plan, img_dtype=torch.uint8, zigzag=zig)
        assert dct.api.last_path() == path
        check_pix("factored", f"{what} inv {src.dtype}{' zz' if zig else ''}", host(got), C, T, Q, random_input=random_input)


@pytest.mark.parametrize("path", ["direct", "tma"])
@pytest.mark.parametrize("qname", QNAMES)
def test_factored_inverse(dct, oracle, qname, path):
    Q, keep = q_of(oracle, qname, dct)
    H, W = 520, 2080
    adv = np.tile(inputs.adversarial(W // 8), (H // 128 + 1, 1))[:H].astype(np.uint8)
    for name, img in (("rand", u8_image(H, W, 11)), ("adversarial", adv),
                      ("smooth", inputs.smooth_image(H, W).astype(np.uint8))):
        run_factored(dct, oracle, img, Q, keep, path, f"{qname} {path} {name}", random_input=name == "rand")


@pytest.mark.parametrize("shape,path", SHAPE_PATHS)
def test_factored_shapes(dct, oracle, shape, path):
    run_factored(dct, oracle, u8_image(*shape, 5), oracle.jpeg_Q(), dct.ALL_COEFFS, path, f"{shape} {path}")


@pytest.mark.parametrize("qname", QNAMES)
def test_factored_families(dct, oracle, qname):
    """Metrics, any-size, batch, host round trip and host pipeline with the factored inverse."""
    T = oracle.haweel_T()
    Q, keep = q_of(oracle, qname, dct)
    H, W = 72, 1056
    imgs = [u8_image(H, W, s) for s in (21, 22, 23)]
    Cs = [oracle.dct(i, Q=Q, keep=keep) for i in imgs]     # the forward chain == the oracle (run_factored)
    plan = factored_plan(dct, Q, keep)
    for img, C in zip(imgs, Cs):
        Y, B = R.forward64(img, T)
        check_coef("factored", f"{qname} families", C, Y, B, Q, keep)
    outs = dct.roundtrip_batch([dev(i) for i in imgs], plan=plan)
    assert dct.api.last_path() == "direct"
    for o, C in zip(outs, Cs):
        check_pix("factored", f"{qname} batch", host(o), C, T, Q)
    d = dev(imgs[0])
    frame = torch.zeros(H + 1, W + 3, dtype=torch.uint8, device="cuda")
    view = frame[1:, 3:]
    view.copy_(d)
    got = dct.roundtrip_any(view, plan=plan)
    assert dct.api.last_path() == "any"
    check_pix("factored", f"{qname} any", host(got), Cs[0], T, Q)
    out, (mse, peen, nnz) = dct.roundtrip_with_metrics(d, plan=plan)
    assert dct.api.last_path() == "direct"
    o = host(out)
    check_pix("factored", f"{qname} metrics", o, Cs[0], T, Q)
    wm, wp = oracle.metrics(imgs[0], o)
    assert mse == pytest.approx(wm, rel=1e-12) and peen == pytest.approx(wp, rel=1e-12)
    assert nnz == int(np.count_nonzero(Cs[0]))
    big = u8_image(520, 2080, 24)
    Cb = oracle.dct(big, Q=Q, keep=keep)
    check_pix("factored", f"{qname} host", dct.roundtrip_host(big, plan=plan), Cb, T, Q)
    res = [np.empty_like(big), np.empty_like(imgs[1])]
    with dct.HostPipeline(plan) as pipe:
        pipe.submit(big, res[0])
        pipe.submit(imgs[1], res[1])
    check_pix("factored", f"{qname} pipeline", res[0], Cb, T, Q)
    check_pix("factored", f"{qname} pipeline", res[1], Cs[1], T, Q)


# ---------------------------------------------------------------- colour: k_rgb / k_rgb_inverse with FINV
def check_rgb(oracle, what, got, coef3, T, Qs):
    """RGB from the kernel against libjpeg's YCbCr -> RGB (the oracle) of the exact planes: at a pixel
    where some plane is ambiguous, any of the (at most 8) combinations of admissible plane values is
    accepted."""
    want, amb, other = [], [], []
    for c in range(3):
        P, Bi = R.inverse64(coef3[c], T, Qs[c])
        w, a, o = R.expected_u8(P, Bi)
        want.append(w), amb.append(a), other.append(o)
    ok = np.zeros(got.shape[:2], bool)
    base = None
    for combo in range(8):
        planes = [np.where(amb[c] & bool(combo >> c & 1), other[c], want[c]) for c in range(3)]
        cand = oracle.ycc_to_rgb(*planes)
        ok |= (cand == got).all(axis=2)
        base = cand if combo == 0 else base
    any_amb = amb[0] | amb[1] | amb[2]
    flips = int(((base != got).any(axis=2)).sum())
    ch = R.Check(int((~ok).sum()), float(any_amb.mean()), 0.0, ok.size)
    print(f"[reassoc] colour {what}: {ch}, pixels on an alternative: {flips}")
    w, a = WORST.get("colour", (0.0, 0.0))
    WORST["colour"] = (w, max(a, ch.ambiguous))
    assert ch.bad == 0, f"colour {what}: {ch}"


@pytest.mark.parametrize("qname", ["jpeg", "jpeg_mask21", "jpeg_x037", "chroma_x2"])
def test_colour(dct, oracle, qname):
    T = oracle.haweel_T()
    Q, keep = q_of(oracle, "jpeg" if qname == "chroma_x2" else qname, dct)
    Qc = oracle.jpeg_Q_chroma()
    Qc = (Qc * F32(0.37)).astype(F32) if qname == "jpeg_x037" else (Qc * F32(2)).astype(F32) if qname == "chroma_x2" else Qc
    plan = dct.Plan(Q=Q, Qc=Qc, keep=keep, inverse=dct.api.INVERSE_FACTORED)
    H, W = 520, 2080
    rng = np.random.default_rng(31)
    rgb = rng.integers(0, 256, (H, W, 3)).astype(np.uint8)
    sm = inputs.smooth_image(H, W)
    rgb[: H // 2] = np.stack([sm, 255 - sm, np.roll(sm, 17, axis=1)], 2)[: H // 2].astype(np.uint8)
    d = dev(rgb)
    streams = dct.forward_rgb(d, plan=plan)
    assert dct.api.last_path() == "rgb"
    planes = oracle.rgb_to_ycc(rgb)
    Qs = (Q, Qc, Qc)
    coef3 = [R.unzigzag(s) for s in host(streams)]
    for c in range(3):
        Y, B = R.forward64(planes[c], T)
        check_coef("colour", f"{qname} plane {c}", coef3[c], Y, B, Qs[c], keep)
    got = dct.inverse_rgb(streams, plan=plan)
    assert dct.api.last_path() == "rgb"
    check_rgb(oracle, f"{qname} split", host(got), coef3, T, Qs)
    zz = torch.empty_like(streams)
    fused = dct.roundtrip_rgb(d, streams=zz, plan=plan)
    assert torch.equal(zz, streams)
    check_rgb(oracle, f"{qname} fused+streams", host(fused), coef3, T, Qs)
    check_rgb(oracle, f"{qname} fused", host(dct.roundtrip_rgb(d, plan=plan)), coef3, T, Qs)


# ---------------------------------------------------------------- tensor-core arm
@pytest.mark.parametrize("shape", [(8, 8), (72, 1056), (520, 2080), (2048, 2048)])
@pytest.mark.parametrize("qname", QNAMES)
@pytest.mark.parametrize("tname", ["dct2", "randsym"])
def test_tensor_core_arm(dct, oracle, tname, qname, shape):
    T = T_of(oracle, tname)
    Q, keep = q_of(oracle, qname, dct)
    img = inputs.float_noise(*shape, 3) if shape[0] % 16 else u8_image(*shape, 9).astype(F32)
    plan = dct.Plan(T=T, Q=Q, keep=keep, dense=dct.api.DENSE_MMA)
    d = dev(img)
    coef = torch.empty_like(d)
    out = dct.roundtrip(d, coef=coef, plan=plan)
    assert dct.api.last_path() == "mma"
    Y, B = R.forward64(img, T)
    C = host(coef)
    what = f"{tname} {qname} {shape}"
    check_coef("mma", what, C, Y, B, Q, keep, R.C_MMA, random_input=True)
    check_pix("mma", what, host(out), C, T, Q, R.C_MMA, random_input=True)
    assert same(dct.roundtrip(d, plan=plan), out)
    if qname == "jpeg":
        check_forward_exact("mma", what, dct, d, Y, B, T, R.C_MMA, dense=dct.api.DENSE_MMA)


def test_tensor_core_scale_sweep(dct, oracle):
    T = oracle.dct2_T()
    rng = np.random.default_rng(21)
    x0 = rng.integers(0, 256, (256, 256)).astype(F32)
    x0[:128] = inputs.adversarial(32)
    for k in SCALES:
        s = F32(2.0 ** k)
        x = (F32(128) + s * (x0 - F32(128))).astype(F32)
        Q = (oracle.jpeg_Q() * s).astype(F32)
        d = dev(x)
        coef = torch.empty_like(d)
        out = dct.roundtrip(d, coef=coef, plan=dct.Plan(T=T, Q=Q, dense=dct.api.DENSE_MMA))
        assert dct.api.last_path() == "mma"
        Y, B = R.forward64(x, T)
        C = host(coef)
        check_coef("mma", f"scale 2^{k}", C, Y, B, Q, dct.ALL_COEFFS, R.C_MMA)
        check_pix("mma", f"scale 2^{k}", host(out), C, T, Q, R.C_MMA)
        check_forward_exact("mma", f"scale 2^{k}", dct, d, Y, B, T, R.C_MMA, dense=dct.api.DENSE_MMA)


# ---------------------------------------------------------------- the defaults are these kernels
@pytest.mark.factored
def test_auto_defaults_resolve_to_the_reassociated_kernels(dct, oracle):
    """With no environment override, AUTO picks the even/odd kernels for a symmetric dense T and the
    factored inverse for u8 output of Haweel's T: same kernels, same bits as the explicit modes."""
    img = u8_image(520, 2080, 41)
    d8, d32 = dev(img), dev(img.astype(F32))
    T = oracle.dct2_T()
    auto = dct.Plan(T=T)
    assert auto.kernel_kind == 2
    for d in (d8, d32):
        for path in (1, 2):
            a = dct.roundtrip(d, plan=dct.Plan(T=T, path=path))
            pa = dct.api.last_path()
            b = dct.roundtrip(d, plan=dct.Plan(T=T, path=path, dense=dct.api.DENSE_SYMMETRIC))
            assert dct.api.last_path() == pa and same(a, b)
    for path in (1, 2):
        a = dct.roundtrip(d8, plan=dct.Plan(path=path))
        pa = dct.api.last_path()
        b = dct.roundtrip(d8, plan=dct.Plan(path=path, inverse=dct.api.INVERSE_FACTORED))
        assert dct.api.last_path() == pa and torch.equal(a, b)
    rgb = torch.from_numpy(np.stack([img, img[::-1], 255 - img], 2).copy()).cuda()
    assert torch.equal(dct.roundtrip_rgb(rgb), dct.roundtrip_rgb(rgb, plan=dct.Plan(inverse=dct.api.INVERSE_FACTORED)))
