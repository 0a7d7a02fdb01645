"""CPU: the 4:2:0 reference (tests/rgb420_ref.py) pinned against the real libjpeg (tests/golden/libjpeg_420.npz,
written by make_libjpeg_420_golden.py), its structure, and a real 4:2:0 JPEG file written around its streams."""
import io
import os

import numpy as np
import pytest

import rgb420_ref as R
from test_color_cpu import BitWriter, huff_codes
from test_gpu_rgb import images

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "libjpeg_420.npz")
ZZ = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
      35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63]


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def test_downsampler_matches_libjpeg(oracle, gold):
    """Groups whose sums are 4k + 2 / 4k + 1 in alternating columns: libjpeg's bias makes them one value, the
    swapped order two.  Every decoded Cb / Cr sample equals the reference's down- then upsampling."""
    for key in ("down", "down_swap"):
        _, cb, cr = oracle.rgb_to_ycc(gold[f"{key}_rgb"])
        for c, p in ((1, cb), (2, cr)):
            half = R.downsample_h2v2(p)
            per_mcu = half.reshape(half.shape[0] // 8, 8, half.shape[1] // 8, 8)
            flat = (per_mcu == per_mcu[:, :1, :, :1]).all()
            assert flat == (key == "down"), f"{key} plane {c}: one value per MCU only in libjpeg's bias order"
            assert np.array_equal(R.upsample_h2v2_fancy(half), gold[f"{key}_ycc"][..., c]), f"{key} plane {c}"


def test_upsampler_matches_libjpeg(oracle, gold):
    """Constant-colour MCUs: the half-resolution planes are libjpeg's, and so is every upsampled sample."""
    _, cb, cr = oracle.rgb_to_ycc(gold["up_rgb"])
    for c, p in ((1, cb), (2, cr)):
        half = R.downsample_h2v2(p)
        assert np.array_equal(half[::8, ::8], gold["up_half"][..., c - 1])
        up = R.upsample_h2v2_fancy(half)
        assert np.count_nonzero(up != np.repeat(np.repeat(half, 2, 0), 2, 1)) > 1000   # the filter is exercised
        assert np.array_equal(up, gold["up_ycc"][..., c]), f"plane {c}"


def test_luma_stream_is_the_444_luma_stream(oracle):
    for Q, Qc, keep in ((None, None, oracle.ALL_COEFFS), (oracle.jpeg_Q() * 0.37, oracle.jpeg_Q_chroma() * 1.3, oracle.zigzag_mask(10))):
        for name, rgb in images((48, 80), 3).items():
            y, cb, cr = R.forward_rgb420(oracle, rgb, Q, Qc, keep)
            _, coef = oracle.roundtrip_rgb(rgb, Q=Q, Qc=Qc, keep=keep, want_coef=True)
            assert np.array_equal(y, oracle.zigzag_i16(coef[0])), name
            assert y.shape == (6, 10, 64) and cb.shape == cr.shape == (3, 5, 64)


def test_grey_image_has_zero_chroma_streams(oracle):
    rng = np.random.default_rng(4)
    grey = np.repeat(rng.integers(0, 256, (32, 48, 1), dtype=np.uint8), 3, 2)
    y, cb, cr = R.forward_rgb420(oracle, grey)
    assert np.count_nonzero(cb) == 0 and np.count_nonzero(cr) == 0 and np.count_nonzero(y) > 0


def write_jpeg_420(streams, H, W, Q, Qc, oracle):
    """A baseline JPEG file around the 4:2:0 streams: SOF0 with three components (sampling 2x2, 1x1, 1x1), Annex K
    tables, and three non-interleaved scans (Y, Cb, Cr), in which each component's blocks come in raster order
    (ITU-T T.81 A.2.2).  Returns the file and the number of entropy-coded bits of the three scans."""
    def seg(marker, payload):
        return bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + bytes(payload)

    f = bytearray(b"\xff\xd8")
    for t, q in ((0, Q), (1, Qc)):
        f += seg(0xDB, bytes([t]) + bytes(int(q[ZZ[k]]) for k in range(64)))
    f += seg(0xC0, bytes([8]) + H.to_bytes(2, "big") + W.to_bytes(2, "big") + bytes([3, 1, 0x22, 0, 2, 0x11, 1, 3, 0x11, 1]))
    codes = {}
    for which in (0, 1):
        for t in (0, 1):
            bits, vals = oracle.huffman_spec(which, t)
            f += seg(0xC4, bytes([(which << 4) | t]) + bytes(bits.tolist()) + bytes(vals.tolist()))
            codes[which, t] = huff_codes(bits, vals)
    total = 0
    for comp, s in enumerate(streams):
        t = 0 if comp == 0 else 1
        dc, ac = codes[0, t], codes[1, t]
        f += seg(0xDA, bytes([1, comp + 1, (t << 4) | t, 0, 63, 0]))
        bw, prev = BitWriter(), 0

        def put_value(v, size):
            if size:
                bw.put(v if v >= 0 else v + (1 << size) - 1, size)

        for blk in s.reshape(-1, 64).astype(int):
            d = int(blk[0]) - prev
            prev = int(blk[0])
            size = abs(d).bit_length()
            bw.put(*dc[size])
            put_value(d, size)
            run = 0
            for k in range(1, 64):
                v = int(blk[k])
                if v == 0:
                    run += 1
                    continue
                while run > 15:
                    bw.put(*ac[0xF0])
                    run -= 16
                size = abs(v).bit_length()
                bw.put(*ac[(run << 4) | size])
                put_value(v, size)
                run = 0
            if run:
                bw.put(*ac[0x00])
        total += bw.bits
        bw.flush()
        f += bw.out
    return bytes(f + b"\xff\xd9"), total


def test_coded_bits_is_the_size_of_a_real_420_jpeg(oracle):
    """libjpeg decodes the 4:2:0 file written around the reference's streams; its entropy-coded bits are the sum of
    the three coded_bits, and its RGB lands near the reference's own 4:2:0 reconstruction."""
    from PIL import Image

    H, W = 48, 80
    yy, xx = np.mgrid[0:H, 0:W]
    rgb = np.stack([128 + 90 * np.sin(xx / 17.0 + c) * np.cos(yy / 13.0 - c) for c in range(3)], -1).clip(0, 255).astype(np.uint8)
    Q, Qc = oracle.jpeg_Q(), oracle.jpeg_Q_chroma()
    streams = R.forward_rgb420(oracle, rgb)
    data, bits = write_jpeg_420(streams, H, W, Q, Qc, oracle)
    assert bits == oracle.coded_bits(streams[0], 0) + oracle.coded_bits(streams[1], 1) + oracle.coded_bits(streams[2], 1)
    im = Image.open(io.BytesIO(data))
    assert im.mode == "RGB" and im.size == (W, H)
    assert [lay[1:3] for lay in im.layer] == [(2, 2), (1, 1), (1, 1)]
    dec = np.array(im).astype(float)
    own = R.inverse_rgb420(oracle, streams).astype(float)
    # Haweel's T approximates the DCT, so libjpeg's exact inverse DCT lands close to the reference's reconstruction
    err = np.mean((dec - own) ** 2)
    print(f"libjpeg decode of the 4:2:0 streams vs own inverse: MSE {err:.1f}; own vs input {np.mean((own - rgb) ** 2):.1f}")
    assert err < 100.0 and np.mean((dec - rgb) ** 2) < 150.0
