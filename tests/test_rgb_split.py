"""The split colour API (b200dct_forward_rgb / b200dct_inverse_rgb: RGB -> three zig-zag coefficient
streams and back) against the oracle and against the fused b200dct_roundtrip_rgb.  Unmarked tests pin
the EXACT inverse (bit-exact against the oracle); `factored` tests run the library default."""
import numpy as np
import pytest
import torch

from test_gpu_rgb import images


def table_cases(oracle, all_coeffs):
    """The Q / Qc / mask combinations of test_gpu_rgb.test_rgb_tables_masks_and_views: a scaled integer
    table, mask 10, non-integer tables (IEEE-division kernels) with mask 21, and extreme tables."""
    return ((oracle.jpeg_Q() * 2, oracle.jpeg_Q_chroma(), all_coeffs),
            (oracle.jpeg_Q(), oracle.jpeg_Q_chroma(), oracle.zigzag_mask(10)),
            (oracle.jpeg_Q() * 0.37, oracle.jpeg_Q_chroma() * 1.3, oracle.zigzag_mask(21)),
            (np.full(64, 1.0, np.float32), np.full(64, 255.0, np.float32), all_coeffs))


def ref_streams(oracle, coef3):
    return np.stack([oracle.zigzag_i16(coef3[c]) for c in range(3)])


def ref_inverse_rgb(oracle, streams, Q=None, Qc=None):
    """Reference decoder of three zig-zag streams: per plane convertToUnsignedChar(idct(stream)) with Q for Y
    and Qc for Cb / Cr, then libjpeg's YCbCr -> RGB."""
    Q = oracle.jpeg_Q() if Q is None else Q
    Qc = oracle.jpeg_Q_chroma() if Qc is None else Qc
    planes = [oracle.to_u8(oracle.idct(oracle.unzigzag_i16(streams[c]), Q=Q if c == 0 else Qc)) for c in range(3)]
    return oracle.ycc_to_rgb(*planes)


def synthetic_streams(H, W, seed):
    """Streams no forward pass produces: random values in +-2048, all-zero blocks, DC-only blocks and
    blocks with one entry at +-32767."""
    rng = np.random.default_rng(seed)
    s = rng.integers(-2048, 2049, (3, H // 8, W // 8, 64)).astype(np.int16)
    blk = s.reshape(3, -1, 64)
    kind = rng.integers(0, 4, blk.shape[:2])
    blk[kind == 1] = 0
    blk[kind == 2, 1:] = 0
    one = np.argwhere(kind == 3)
    blk[kind == 3] = 0
    pos = rng.integers(0, 64, len(one))
    blk[one[:, 0], one[:, 1], pos] = rng.choice(np.array([-32767, 32767], np.int16), len(one))
    blk[0, 0, 0] = 32767                       # a DC-only block at the extreme, in every shape
    blk[0, 0, 1:] = 0
    return s


def test_reference_decoder_is_the_oracle_round_trip(oracle):
    """Pins ref_inverse_rgb: on the oracle's own coefficient streams it gives oracle.roundtrip_rgb, bit for bit."""
    for Q, Qc in ((None, None), (oracle.jpeg_Q() * 0.37, oracle.jpeg_Q_chroma() * 1.3)):
        for name, rgb in images((64, 96), 3).items():
            want, coef = oracle.roundtrip_rgb(rgb, Q=Q, Qc=Qc, want_coef=True)
            assert np.array_equal(ref_inverse_rgb(oracle, ref_streams(oracle, coef), Q, Qc), want), name


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(8, 8), (64, 96), (256, 256), (520, 1064)])
def test_forward_rgb_matches_oracle(dct, oracle, shape):
    for name, rgb in images(shape, 3).items():
        _, coef = oracle.roundtrip_rgb(rgb, want_coef=True)
        d = torch.from_numpy(rgb).cuda()
        zz = dct.forward_rgb(d)
        assert dct.api.last_launch_count() == 1 and dct.api.last_path() == "rgb"
        assert tuple(zz.shape) == (3, shape[0] // 8, shape[1] // 8, 64) and zz.dtype == torch.int16
        assert np.array_equal(zz.cpu().numpy(), ref_streams(oracle, coef)), name
        assert np.array_equal(d.cpu().numpy(), rgb), f"{name}: input modified"


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(8, 8), (64, 96), (256, 256), (520, 1064)])
def test_inverse_rgb_matches_oracle(dct, oracle, shape):
    H, W = shape
    for name, rgb in images(shape, 5).items():
        want, coef = oracle.roundtrip_rgb(rgb, want_coef=True)
        streams = ref_streams(oracle, coef)
        d = torch.from_numpy(streams).cuda()
        out = dct.inverse_rgb(d)
        assert dct.api.last_launch_count() == 1 and dct.api.last_path() == "rgb"
        assert tuple(out.shape) == (H, W, 3) and out.dtype == torch.uint8
        assert np.array_equal(out.cpu().numpy(), want), name
        assert np.array_equal(d.cpu().numpy(), streams), f"{name}: streams modified"
    s = synthetic_streams(H, W, 7)
    out = dct.inverse_rgb(torch.from_numpy(s).cuda())
    assert np.array_equal(out.cpu().numpy(), ref_inverse_rgb(oracle, s)), "synthetic streams"


def _split_equals_fused(dct, oracle):
    for Q, Qc, keep in table_cases(oracle, dct.ALL_COEFFS):
        plan = dct.Plan(Q=Q, Qc=Qc, keep=keep)
        for name, rgb in images((136, 264), 9).items():
            x = torch.from_numpy(rgb).cuda()
            fused_zz = torch.empty(3, 17, 33, 64, dtype=torch.int16, device="cuda")
            fused = dct.roundtrip_rgb(x, streams=fused_zz, plan=plan)
            zz = dct.forward_rgb(x, plan=plan)
            assert torch.equal(zz, fused_zz), name
            assert torch.equal(dct.inverse_rgb(zz, plan=plan), fused), name
            assert torch.equal(dct.roundtrip_rgb(x, plan=plan), fused), name


@pytest.mark.gpu
def test_split_equals_fused(dct, oracle):
    _split_equals_fused(dct, oracle)


@pytest.mark.gpu
@pytest.mark.factored
def test_split_equals_fused_default_inverse(dct, oracle):
    _split_equals_fused(dct, oracle)


@pytest.mark.gpu
def test_split_rgb_views_and_padded_planes(dct, oracle):
    """A window of a larger image in, streams whose planes lie further apart than needed, a window of a
    frame out: nothing outside the described bytes is written."""
    big = torch.from_numpy(images((128, 256), 4)["smooth"]).cuda()
    src = big[16:80, 32:160]
    H, W = 64, 128
    want, coef = oracle.roundtrip_rgb(src.cpu().numpy(), want_coef=True)
    buf = torch.full((3, H // 8 + 1, W // 8, 64), -12345, dtype=torch.int16, device="cuda")
    streams = buf[:, : H // 8]                  # plane stride (H/8 + 1) block-rows
    assert dct.forward_rgb(src, streams=streams) is streams
    assert np.array_equal(streams.cpu().numpy(), ref_streams(oracle, coef))
    assert bool((buf[:, H // 8] == -12345).all()), "gap between planes written"
    frame = torch.full((128, 256, 3), 77, dtype=torch.uint8, device="cuda")
    dst = frame[8:72, 64:192]
    assert dct.inverse_rgb(streams, out=dst) is dst
    assert np.array_equal(dst.cpu().numpy(), want)
    mask = torch.ones(128, 256, dtype=torch.bool, device="cuda")
    mask[8:72, 64:192] = False
    assert bool((frame[mask] == 77).all()), "frame outside the window written"


@pytest.mark.gpu
def test_split_rgb_argument_errors(dct, oracle):
    ARG, SHAPE, ALIGN = -1, -2, -3
    rgb = torch.zeros(16, 16, 3, dtype=torch.uint8, device="cuda")
    zz = torch.zeros(3, 2, 2, 64, dtype=torch.int16, device="cuda")
    dense = dct.Plan(T=oracle.dct2_T())
    with pytest.raises(dct.B200DCTError):
        dct.forward_rgb(rgb, plan=dense)                                               # Haweel's T only
    with pytest.raises(dct.B200DCTError):
        dct.inverse_rgb(zz, plan=dense)
    with pytest.raises(dct.B200DCTError):
        dct.forward_rgb(torch.zeros(16, 12, 3, dtype=torch.uint8, device="cuda"))      # W % 8
    with pytest.raises(dct.B200DCTError):
        dct.forward_rgb(torch.zeros(16, 16, 3, device="cuda"))                         # f32
    with pytest.raises(dct.B200DCTError):
        dct.inverse_rgb(zz.float())
    with pytest.raises(dct.B200DCTError):
        dct.inverse_rgb(zz, out=torch.zeros(16, 16, 3, device="cuda"))
    with pytest.raises(dct.B200DCTError):
        dct.forward_rgb(rgb, streams=torch.zeros(3, 2, 2, 32, dtype=torch.int16, device="cuda"))
    with pytest.raises(dct.B200DCTError):
        dct.inverse_rgb(zz, out=torch.zeros(16, 8, 3, dtype=torch.uint8, device="cuda"))
    # the C ABI directly, where the wrapper would reject the case first
    good = dct.Plan()
    L, h, plane = dct.lib(), good._h, zz.stride(0) * 2
    buf = torch.zeros(64, 64, dtype=torch.uint8, device="cuda")      # room for every pitch below
    p, z = buf.data_ptr(), zz.data_ptr()
    fwd = lambda *a: L.b200dct_forward_rgb(*a, None)
    inv = lambda *a: L.b200dct_inverse_rgb(*a, None)
    assert fwd(h, p, 48, z, plane, 16, 16) == 0 and inv(h, z, plane, p, 48, 16, 16) == 0
    torch.cuda.synchronize()
    cases = [
        (fwd(None, p, 48, z, plane, 16, 16), ARG), (fwd(h, None, 48, z, plane, 16, 16), ARG), (fwd(h, p, 48, None, plane, 16, 16), ARG),
        (inv(None, z, plane, p, 48, 16, 16), ARG), (inv(h, None, plane, p, 48, 16, 16), ARG), (inv(h, z, plane, None, 48, 16, 16), ARG),
        (fwd(dense._h, p, 48, z, plane, 16, 16), ARG), (inv(dense._h, z, plane, p, 48, 16, 16), ARG),
        (fwd(h, p, 48, z, plane, 16, 12), SHAPE), (inv(h, z, plane, p, 48, 12, 16), SHAPE), (fwd(h, p, 48, z, plane, 0, 16), SHAPE),
        (fwd(h, p, 40, z, plane, 16, 16), SHAPE), (inv(h, z, plane, p, 40, 16, 16), SHAPE),          # pitch < W * 3
        (fwd(h, p + 1, 48, z, plane, 16, 16), ALIGN), (inv(h, z, plane, p + 4, 48, 16, 16), ALIGN),  # pixel pointer
        (fwd(h, p, 52, z, plane, 16, 16), ALIGN), (inv(h, z, plane, p, 52, 16, 16), ALIGN),          # pixel pitch
        (fwd(h, p, 48, z + 8, plane, 16, 16), ALIGN), (inv(h, z + 8, plane, p, 48, 16, 16), ALIGN),  # stream pointer
        (fwd(h, p, 48, z, plane - 16, 16, 16), ALIGN), (inv(h, z, plane - 16, p, 48, 16, 16), ALIGN),  # planes overlap
        (fwd(h, p, 48, z, plane + 8, 16, 16), ALIGN), (inv(h, z, plane + 8, p, 48, 16, 16), ALIGN),
    ]
    for k, (rc, want) in enumerate(cases):
        assert rc == want, f"case {k}: {rc} != {want}"
    assert dct.api.last_launch_count() == 0 and dct.api.last_path() == "none"


@pytest.mark.gpu
def test_split_rgb_stream_order_and_early_path(dct, oracle):
    """The split calls take part in the early-load protocol (see early loads, b200dct.cu).  4096^2 RGB is 2048
    CTAs, more than the machine holds at once, so a call whose input the library's previous launch does not
    write loads before that launch has completed.  Foreign kernels that write the next call's input, calls that
    read what the previous call (or the one before it) wrote, and independent calls back to back: 30
    iterations without a host synchronisation, every result compared on the device."""
    N = 4096
    plan = dct.Plan()
    grey_plan = dct.Plan(path=dct.api.PATH_DIRECT)       # direct family: a predecessor the colour kernels may overlap
    g = torch.Generator(device="cuda").manual_seed(11)
    src = [torch.randint(0, 256, (N, N, 3), device="cuda", generator=g, dtype=torch.int32).to(torch.uint8) for _ in range(3)]
    grey = [a[..., 1].contiguous() for a in src]
    want_zz = [dct.forward_rgb(a, plan=plan).clone() for a in src]
    want = [dct.roundtrip_rgb(a, plan=plan).clone() for a in src]
    want_grey = [dct.roundtrip(a, plan=grey_plan).clone() for a in grey]
    want2 = dct.roundtrip_rgb(want[0], plan=plan).clone()
    torch.cuda.synchronize()
    band = src[0][:16].cpu().numpy()
    want_band, coef_band = oracle.roundtrip_rgb(band, want_coef=True)
    assert np.array_equal(want[0][:16].cpu().numpy(), want_band)
    assert np.array_equal(want_zz[0][:, :2].cpu().numpy(), ref_streams(oracle, coef_band))

    bad = torch.zeros((), dtype=torch.int64, device="cuda")

    def check(a, b):
        bad.add_((a != b).sum())

    x = torch.empty_like(src[0])
    zz = [torch.empty_like(want_zz[0]) for _ in range(2)]
    outs = [torch.empty_like(x) for _ in range(2)]
    rts = [torch.empty_like(x) for _ in range(2)]
    gouts = [torch.empty_like(grey[0]) for _ in range(2)]
    for it in range(30):
        k, j = it % 3, it % 2
        x.copy_(src[k])                                          # a foreign kernel writes the input of the next call
        dct.forward_rgb(x, streams=zz[j], plan=plan)
        if it % 5 == 4:
            x.fill_(0)                                           # and clobbers it right behind the call
        dct.roundtrip(grey[k], out=gouts[j], plan=grey_plan)     # independent of the forward pass
        dct.inverse_rgb(zz[j], out=outs[j], plan=plan)           # reads what the launch before last wrote
        dct.roundtrip_rgb(src[k], out=rts[j], plan=plan)         # independent of the inverse pass
        check(zz[j], want_zz[k])
        check(outs[j], want[k])
        check(rts[j], want[k])
        check(gouts[j], want_grey[k])
    # dependent chain: every call reads what its predecessor wrote, the last one overwrites what its predecessor reads
    a, b, za, zb = torch.empty_like(x), torch.empty_like(x), torch.empty_like(zz[0]), torch.empty_like(zz[0])
    for rep in range(10):
        dct.forward_rgb(src[0], streams=za, plan=plan)
        dct.inverse_rgb(za, out=a, plan=plan)
        dct.forward_rgb(a, streams=zb, plan=plan)
        dct.inverse_rgb(zb, out=b, plan=plan)
        dct.forward_rgb(src[1], streams=zb, plan=plan)
    check(za, want_zz[0])
    check(a, want[0])
    check(b, want2)
    check(zb, want_zz[1])
    # independent calls back to back (the early path proper)
    fz, io = [torch.empty_like(zz[0]) for _ in range(3)], [torch.empty_like(x) for _ in range(3)]
    for rep in range(10):
        for i in range(3):
            dct.forward_rgb(src[i], streams=fz[i], plan=plan)
            dct.inverse_rgb(want_zz[i], out=io[i], plan=plan)
    for i in range(3):
        check(fz[i], want_zz[i])
        check(io[i], want[i])
    torch.cuda.synchronize()
    assert int(bad.item()) == 0


@pytest.mark.gpu
def test_split_rgb_graph_capture(dct, oracle):
    rgb = torch.from_numpy(images((256, 512), 2)["smooth"]).cuda()
    plan = dct.Plan()
    want_zz = dct.forward_rgb(rgb, plan=plan).clone()
    want = dct.inverse_rgb(want_zz, plan=plan).clone()
    torch.cuda.synchronize()
    zz, out = torch.zeros_like(want_zz), torch.zeros_like(rgb)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.graph(g, stream=s):
        dct.forward_rgb(rgb, streams=zz, plan=plan, stream=torch.cuda.current_stream())
        dct.inverse_rgb(zz, out=out, plan=plan, stream=torch.cuda.current_stream())
    for _ in range(3):
        zz.zero_()
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(zz, want_zz) and torch.equal(out, want)
    assert np.array_equal(want.cpu().numpy(), oracle.roundtrip_rgb(rgb.cpu().numpy()))
