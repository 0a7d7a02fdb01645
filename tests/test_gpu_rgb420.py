"""GPU: the 4:2:0 colour calls (b200dct_forward_rgb420 / b200dct_inverse_rgb420) against the CPU reference
(tests/rgb420_ref.py, pinned against the real libjpeg by tests/test_rgb420_cpu.py).  Unmarked tests pin the EXACT
inverse (bit-exact RGB); the `factored` test holds the library default to the float64 criterion of f64ref.py."""
import numpy as np
import pytest
import torch

import f64ref as F
import rgb420_ref as R
from test_gpu_rgb import images

pytestmark = pytest.mark.gpu

# 16 x 16 .. non-square with partial CTA tiles in both dimensions (forward: 16 x 2 MCUs per CTA; inverse: 32 x 4)
SHAPES = [(16, 16), (16, 80), (48, 16), (48, 80), (272, 1072)]


def dev(streams):
    return tuple(torch.from_numpy(np.ascontiguousarray(s)).cuda() for s in streams)


def host(streams):
    return tuple(s.cpu().numpy() for s in streams)


def table_cases(oracle, all_coeffs):
    """The quantiser variants of test_rgb_split: Q x 2, mask 10, and non-integer tables (the __fdiv_rn kernels)."""
    return ((oracle.jpeg_Q() * 2, oracle.jpeg_Q_chroma(), all_coeffs),
            (oracle.jpeg_Q(), oracle.jpeg_Q_chroma(), oracle.zigzag_mask(10)),
            (oracle.jpeg_Q() * 0.37, oracle.jpeg_Q_chroma() * 1.3, oracle.zigzag_mask(21)))


def sparse_streams(H, W, seed):
    """Streams no forward pass produces: sparse random values in +-2048, all-zero, DC-only and +-32767 blocks, so
    that own, halo and edge chroma samples take arbitrary values."""
    rng = np.random.default_rng(seed)
    out = []
    for h, w in ((H // 8, W // 8), (H // 16, W // 16), (H // 16, W // 16)):
        s = rng.integers(-2048, 2049, (h, w, 64)) * (rng.random((h, w, 64)) < 0.15)
        blk = s.reshape(-1, 64)
        kind = rng.integers(0, 4, len(blk))
        blk[kind == 1] = 0
        blk[kind == 2, 1:] = 0
        blk[kind == 3] = 0
        blk[kind == 3, rng.integers(0, 64)] = 32767
        out.append(s.astype(np.int16))
    return tuple(out)


@pytest.mark.parametrize("shape", SHAPES)
def test_forward_rgb420_matches_reference(dct, oracle, shape):
    H, W = shape
    for name, rgb in images(shape, 3).items():
        d = torch.from_numpy(rgb).cuda()
        y, cb, cr = dct.forward_rgb420(d)
        assert dct.api.last_launch_count() == 1 and dct.api.last_path() == "rgb"
        assert tuple(y.shape) == (H // 8, W // 8, 64) and tuple(cb.shape) == tuple(cr.shape) == (H // 16, W // 16, 64)
        want = R.forward_rgb420(oracle, rgb)
        for c, (g, w) in enumerate(zip(host((y, cb, cr)), want)):
            assert np.array_equal(g, w), f"{name} plane {c}"
        assert torch.equal(y, dct.forward_rgb(d)[0]), f"{name}: Y stream differs from forward_rgb's"
        assert np.array_equal(d.cpu().numpy(), rgb), f"{name}: input modified"


def test_forward_rgb420_quantiser_variants(dct, oracle):
    rgb = images((80, 208), 9)
    for Q, Qc, keep in table_cases(oracle, dct.ALL_COEFFS):
        plan = dct.Plan(Q=Q, Qc=Qc, keep=keep)
        for name, x in rgb.items():
            got = host(dct.forward_rgb420(torch.from_numpy(x).cuda(), plan=plan))
            for c, (g, w) in enumerate(zip(got, R.forward_rgb420(oracle, x, Q, Qc, keep))):
                assert np.array_equal(g, w), f"{name} plane {c}"
            # and their exact inverse
            out = dct.inverse_rgb420(dev(got), plan=plan)
            assert np.array_equal(out.cpu().numpy(), R.inverse_rgb420(oracle, got, Q, Qc)), name


@pytest.mark.parametrize("shape", SHAPES)
def test_inverse_rgb420_matches_reference(dct, oracle, shape):
    H, W = shape
    for name, rgb in images(shape, 5).items():
        streams = R.forward_rgb420(oracle, rgb)
        d = dev(streams)
        out = dct.inverse_rgb420(d)
        assert dct.api.last_launch_count() == 1 and dct.api.last_path() == "rgb"
        assert tuple(out.shape) == (H, W, 3) and out.dtype == torch.uint8
        assert np.array_equal(out.cpu().numpy(), R.inverse_rgb420(oracle, streams)), name
        assert all(np.array_equal(g, w) for g, w in zip(host(d), streams)), f"{name}: streams modified"
    s = sparse_streams(H, W, 7)
    out = dct.inverse_rgb420(dev(s))
    assert np.array_equal(out.cpu().numpy(), R.inverse_rgb420(oracle, s)), "synthetic streams"


def check_factored(oracle, got, streams, Q, Qc):
    """RGB of the factored inverse against exact arithmetic.  Every decoded plane sample is either fixed or one of
    two admissible values (f64ref.expected_u8 on the float64 inverse of the kernel's own coefficients).  The
    upsampling weights are positive and R, G, B are each monotone in Y, Cb and Cr, so every output channel must
    lie between its values at the extreme combinations -- and be exact where no contributing sample is ambiguous."""
    T = oracle.haweel_T()
    lohi = []
    for c, (s, q) in enumerate(zip(streams, (Q, Qc, Qc))):
        P, Bi = F.inverse64(F.unzigzag(s), T, q)
        want, amb, other = F.expected_u8(P, Bi)
        lo, hi = np.minimum(want, other), np.maximum(want, other)
        lohi.append((lo, hi) if c == 0 else (R.upsample_h2v2_fancy(lo), R.upsample_h2v2_fancy(hi)))
    cands = np.stack([oracle.ycc_to_rgb(*(lohi[c][combo >> c & 1] for c in range(3))) for combo in range(8)])
    lo, hi = cands.min(0), cands.max(0)
    bad = int(((got < lo) | (got > hi)).sum())
    print(f"[factored 4:2:0] channels with an admissible range: {float((lo != hi).mean()):.2e}, off the range: {bad}")
    assert bad == 0


@pytest.mark.factored
@pytest.mark.parametrize("q", ["jpeg", "x037"])
def test_inverse_rgb420_default_mode_within_float64_bound(dct, oracle, q):
    Q, Qc = oracle.jpeg_Q(), oracle.jpeg_Q_chroma()
    if q == "x037":
        Q, Qc = (Q * np.float32(0.37)).astype(np.float32), (Qc * np.float32(1.3)).astype(np.float32)
    plan = dct.Plan(Q=Q, Qc=Qc)
    H, W = 272, 1072
    for name, rgb in images((H, W), 11).items():
        streams = dct.forward_rgb420(torch.from_numpy(rgb).cuda(), plan=plan)
        got = dct.inverse_rgb420(streams, plan=plan)
        check_factored(oracle, got.cpu().numpy(), host(streams), Q, Qc)
    s = sparse_streams(H, W, 13)
    check_factored(oracle, dct.inverse_rgb420(dev(s), plan=plan).cpu().numpy(), s, Q, Qc)


def test_rgb420_pitched_views_and_sentinels(dct, oracle):
    """A window of a larger image in, a window of a frame out: nothing outside the described bytes is written."""
    big = torch.from_numpy(images((128, 256), 4)["smooth"]).cuda()
    src = big[16:80, 32:160]
    H, W = 64, 128
    want = R.forward_rgb420(oracle, src.cpu().numpy())
    pad = torch.full((3, H * W // 64 * 64 + 256), -12345, dtype=torch.int16, device="cuda")
    streams = (pad[0, 128:128 + H * W].view(H // 8, W // 8, 64), pad[1, 128:128 + H * W // 4].view(H // 16, W // 16, 64),
               pad[2, 128:128 + H * W // 4].view(H // 16, W // 16, 64))
    got = dct.forward_rgb420(src, streams=streams)
    assert all(g is s for g, s in zip(got, streams))
    assert all(np.array_equal(g, w) for g, w in zip(host(streams), want))
    for c, n in enumerate((H * W, H * W // 4, H * W // 4)):
        assert bool((pad[c, :128] == -12345).all()) and bool((pad[c, 128 + n:] == -12345).all()), f"stream {c}: outside written"
    frame = torch.full((128, 256, 3), 77, dtype=torch.uint8, device="cuda")
    dst = frame[8:72, 64:192]
    assert dct.inverse_rgb420(streams, out=dst) is dst
    assert np.array_equal(dst.cpu().numpy(), R.inverse_rgb420(oracle, want))
    mask = torch.ones(128, 256, dtype=torch.bool, device="cuda")
    mask[8:72, 64:192] = False
    assert bool((frame[mask] == 77).all()), "frame outside the window written"


def test_rgb420_argument_errors(dct, oracle):
    ARG, SHAPE, ALIGN = -1, -2, -3
    rgb = torch.zeros(32, 32, 3, dtype=torch.uint8, device="cuda")
    zs = dct.forward_rgb420(rgb)
    dense = dct.Plan(T=oracle.dct2_T())
    bad_calls = [
        lambda: dct.forward_rgb420(rgb, plan=dense),                                        # Haweel's T only
        lambda: dct.inverse_rgb420(zs, plan=dense),
        lambda: dct.forward_rgb420(torch.zeros(32, 24, 3, dtype=torch.uint8, device="cuda")),  # W % 16
        lambda: dct.forward_rgb420(torch.zeros(24, 32, 3, dtype=torch.uint8, device="cuda")),  # H % 16
        lambda: dct.forward_rgb420(torch.zeros(32, 32, 3, device="cuda")),                  # f32 pixels
        lambda: dct.inverse_rgb420(zs[:2]),                                                 # two streams
        lambda: dct.inverse_rgb420((zs[0], zs[1], zs[2].float())),
        lambda: dct.inverse_rgb420((zs[0], zs[1], zs[1][:1])),                              # chroma shape
        lambda: dct.inverse_rgb420((zs[0], zs[1].transpose(0, 1), zs[2])),                  # not tightly packed
        lambda: dct.inverse_rgb420(zs, out=torch.zeros(32, 32, 3, device="cuda")),
        lambda: dct.inverse_rgb420(zs, out=torch.zeros(32, 16, 3, dtype=torch.uint8, device="cuda")),
        lambda: dct.forward_rgb420(rgb, streams=(zs[0], zs[1], torch.zeros(2, 2, 32, dtype=torch.int16, device="cuda"))),
    ]
    for call in bad_calls:
        with pytest.raises(dct.B200DCTError):
            call()
    # the C ABI directly, where the wrapper would reject the case first
    good = dct.Plan()
    L, h = dct.lib(), good._h
    buf = torch.zeros(128, 128, dtype=torch.uint8, device="cuda")    # room for every pitch below
    zbuf = torch.zeros(4096, dtype=torch.int16, device="cuda")
    p, y, b, r = buf.data_ptr(), zbuf.data_ptr(), zbuf.data_ptr() + 2048, zbuf.data_ptr() + 4096
    fwd = lambda *a: L.b200dct_forward_rgb420(*a, None)          # noqa: E731  (plan, rgb, pitch, y, cb, cr, H, W)
    inv = lambda *a: L.b200dct_inverse_rgb420(*a, None)          # noqa: E731  (plan, y, cb, cr, out, pitch, H, W)
    assert fwd(h, p, 96, y, b, r, 32, 32) == 0 and inv(h, y, b, r, p, 96, 32, 32) == 0
    torch.cuda.synchronize()
    cases = [
        (fwd(None, p, 96, y, b, r, 32, 32), ARG), (fwd(h, None, 96, y, b, r, 32, 32), ARG), (fwd(h, p, 96, None, b, r, 32, 32), ARG),
        (fwd(h, p, 96, y, None, r, 32, 32), ARG), (fwd(h, p, 96, y, b, None, 32, 32), ARG),
        (inv(None, y, b, r, p, 96, 32, 32), ARG), (inv(h, None, b, r, p, 96, 32, 32), ARG), (inv(h, y, None, r, p, 96, 32, 32), ARG),
        (inv(h, y, b, None, p, 96, 32, 32), ARG), (inv(h, y, b, r, None, 96, 32, 32), ARG),
        (fwd(dense._h, p, 96, y, b, r, 32, 32), ARG), (inv(dense._h, y, b, r, p, 96, 32, 32), ARG),
        (fwd(h, p, 96, y, b, r, 32, 24), SHAPE), (fwd(h, p, 96, y, b, r, 8, 32), SHAPE), (inv(h, y, b, r, p, 96, 24, 32), SHAPE),
        (fwd(h, p, 96, y, b, r, 0, 32), SHAPE), (inv(h, y, b, r, p, 96, 32, -16), SHAPE),
        (fwd(h, p, 88, y, b, r, 32, 32), SHAPE), (inv(h, y, b, r, p, 88, 32, 32), SHAPE),           # pitch < W * 3
        (fwd(h, p + 4, 96, y, b, r, 32, 32), ALIGN), (inv(h, y, b, r, p + 1, 96, 32, 32), ALIGN),   # pixel pointer
        (fwd(h, p, 100, y, b, r, 32, 32), ALIGN), (inv(h, y, b, r, p, 100, 32, 32), ALIGN),         # pixel pitch
        (fwd(h, p, 96, y + 8, b, r, 32, 32), ALIGN), (fwd(h, p, 96, y, b + 2, r, 32, 32), ALIGN),   # stream pointers
        (fwd(h, p, 96, y, b, r + 8, 32, 32), ALIGN), (inv(h, y + 2, b, r, p, 96, 32, 32), ALIGN),
        (inv(h, y, b + 8, r, p, 96, 32, 32), ALIGN), (inv(h, y, b, r + 4, p, 96, 32, 32), ALIGN),
    ]
    for k, (rc, want) in enumerate(cases):
        assert rc == want, f"case {k}: {rc} != {want}"
    assert dct.api.last_launch_count() == 0 and dct.api.last_path() == "none"


def test_rgb420_stream_order_and_early_path(dct, oracle):
    """The 4:2:0 calls take part in the early-load protocol (see early loads, b200dct.cu).  At 8192^2 both kernels
    have more CTAs than the machine holds at once (forward 8192, inverse 2048), so a call whose input the library's
    previous launch does not write loads before that launch has completed.  Foreign kernels that write the next
    call's input, calls that read what the previous call (or the one before it) wrote, and independent calls back
    to back, without a host synchronisation; every result compared on the device."""
    N = 8192
    plan = dct.Plan()
    grey_plan = dct.Plan(path=dct.api.PATH_DIRECT)       # direct family: a predecessor the colour kernels may overlap
    g = torch.Generator(device="cuda").manual_seed(11)
    src = [torch.randint(0, 256, (N, N, 3), device="cuda", generator=g, dtype=torch.int32).to(torch.uint8) for _ in range(3)]
    grey = [a[..., 1].contiguous() for a in src]
    want_zz = [tuple(s.clone() for s in dct.forward_rgb420(a, plan=plan)) for a in src]
    want = [dct.inverse_rgb420(z, plan=plan).clone() for z in want_zz]
    want_grey = [dct.roundtrip(a, plan=grey_plan).clone() for a in grey]
    want2 = dct.inverse_rgb420(dct.forward_rgb420(want[0], plan=plan), plan=plan).clone()
    torch.cuda.synchronize()
    band = src[0][:32].cpu().numpy()                       # the top MCU row depends on the 32 rows above the next one
    band_zz = R.forward_rgb420(oracle, band)
    assert np.array_equal(want_zz[0][0][:2].cpu().numpy(), band_zz[0][:2])
    assert np.array_equal(want_zz[0][1][:1].cpu().numpy(), band_zz[1][:1])
    assert np.array_equal(want[0][:16].cpu().numpy(), R.inverse_rgb420(oracle, band_zz)[:16])

    bad = torch.zeros((), dtype=torch.int64, device="cuda")

    def check(a, b):
        if isinstance(a, tuple):
            for u, v in zip(a, b):
                bad.add_((u != v).sum())
        else:
            bad.add_((a != b).sum())

    def like(z):
        return tuple(torch.empty_like(s) for s in z)

    x = torch.empty_like(src[0])
    zz = [like(want_zz[0]) for _ in range(2)]
    outs = [torch.empty_like(x) for _ in range(2)]
    gouts = [torch.empty_like(grey[0]) for _ in range(2)]
    for it in range(12):
        k, j = it % 3, it % 2
        x.copy_(src[k])                                          # a foreign kernel writes the input of the next call
        dct.forward_rgb420(x, streams=zz[j], plan=plan)
        if it % 5 == 4:
            x.fill_(0)                                           # and clobbers it right behind the call
        dct.roundtrip(grey[k], out=gouts[j], plan=grey_plan)     # independent of the forward pass
        dct.inverse_rgb420(zz[j], out=outs[j], plan=plan)        # reads what the launch before last wrote
        check(zz[j], want_zz[k])
        check(outs[j], want[k])
        check(gouts[j], want_grey[k])
    # dependent chain: every call reads what its predecessor wrote, the last one overwrites what its predecessor reads
    a, b, za, zb = torch.empty_like(x), torch.empty_like(x), like(zz[0]), like(zz[0])
    for rep in range(4):
        dct.forward_rgb420(src[0], streams=za, plan=plan)
        dct.inverse_rgb420(za, out=a, plan=plan)
        dct.forward_rgb420(a, streams=zb, plan=plan)
        dct.inverse_rgb420(zb, out=b, plan=plan)
        dct.forward_rgb420(src[1], streams=zb, plan=plan)
    check(za, want_zz[0])
    check(a, want[0])
    check(b, want2)
    check(zb, want_zz[1])
    # independent calls back to back (the early path proper)
    fz, io = [like(zz[0]) for _ in range(3)], [torch.empty_like(x) for _ in range(3)]
    for rep in range(4):
        for i in range(3):
            dct.forward_rgb420(src[i], streams=fz[i], plan=plan)
            dct.inverse_rgb420(want_zz[i], out=io[i], plan=plan)
    for i in range(3):
        check(fz[i], want_zz[i])
        check(io[i], want[i])
    torch.cuda.synchronize()
    assert int(bad.item()) == 0


def test_rgb420_graph_capture(dct, oracle):
    rgb = torch.from_numpy(images((256, 512), 2)["smooth"]).cuda()
    plan = dct.Plan()
    want_zz = tuple(s.clone() for s in dct.forward_rgb420(rgb, plan=plan))
    want = dct.inverse_rgb420(want_zz, plan=plan).clone()
    torch.cuda.synchronize()
    zz, out = tuple(torch.zeros_like(s) for s in want_zz), torch.zeros_like(rgb)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.graph(g, stream=s):
        dct.forward_rgb420(rgb, streams=zz, plan=plan, stream=torch.cuda.current_stream())
        dct.inverse_rgb420(zz, out=out, plan=plan, stream=torch.cuda.current_stream())
    for _ in range(3):
        for t in zz:
            t.zero_()
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(zz, want_zz)) and torch.equal(out, want)
    assert np.array_equal(want.cpu().numpy(), R.inverse_rgb420(oracle, R.forward_rgb420(oracle, rgb.cpu().numpy())))


def test_rgb420_coded_bits_and_compression_factor(dct, oracle):
    H, W = 272, 1072
    rgb = images((H, W), 6)["smooth"]
    d = torch.from_numpy(rgb).cuda()
    y, cb, cr = dct.forward_rgb420(d)
    ref = R.forward_rgb420(oracle, rgb)
    bits = [dct.coded_bits(s, 0 if c == 0 else 1) for c, s in enumerate((y, cb, cr))]
    assert bits == [oracle.coded_bits(s, 0 if c == 0 else 1) for c, s in enumerate(ref)]
    cf = dct.compression_factor((y, cb, cr))
    assert cf == 8.0 * 3 * H * W / sum(bits)
    # half the coefficients of 4:4:4: the 4:2:0 image codes smaller than the 4:4:4 one of the same pixels
    assert cf > dct.compression_factor(dct.forward_rgb(d))
