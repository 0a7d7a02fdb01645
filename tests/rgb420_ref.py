"""CPU reference of the 4:2:0 colour path (b200dct_forward_rgb420 / b200dct_inverse_rgb420), built on the
oracle's pinned pieces: libjpeg's colour conversions (oracle.rgb_to_ycc / ycc_to_rgb) and the per-plane u8
pipeline (convertToFloat, dct, quantise; dequantise, idct, convertToUnsignedChar).  The two resamplers are
libjpeg's and are pinned against the real libjpeg by tests/golden/libjpeg_420.npz
(tests/golden/make_libjpeg_420_golden.py)."""
import numpy as np


def downsample_h2v2(plane: np.ndarray) -> np.ndarray:
    """jcsample.c h2v2_downsample: (a + b + c + d + bias) >> 2 over each 2x2 group of 8-bit samples, bias 1 at
    even output columns and 2 at odd ones."""
    p = plane.astype(np.int32)
    s = p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2]
    bias = np.tile(np.array([1, 2], np.int32), s.shape[1] // 2 + 1)[: s.shape[1]]
    return ((s + bias) >> 2).astype(np.uint8)


def upsample_h2v2_fancy(plane: np.ndarray) -> np.ndarray:
    """jdsample.c h2v2_fancy_upsample: the half-resolution plane c, edge-replicated on all four sides;
    colsum = 3 c[y] + c[y -+ 1] (row above for the upper output row of a pair, below for the lower one); left
    output pixel (3 colsum[x] + colsum[x - 1] + 8) >> 4, right one (3 colsum[x] + colsum[x + 1] + 7) >> 4."""
    c = np.pad(plane.astype(np.int32), 1, mode="edge")
    h, w = plane.shape
    out = np.empty((2 * h, 2 * w), np.int32)
    for half, nb in ((0, c[0:h]), (1, c[2:h + 2])):
        cs = 3 * c[1:h + 1] + nb                     # (h, w + 2): colsum with a replicated column on each side
        out[half::2, 0::2] = (3 * cs[:, 1:w + 1] + cs[:, 0:w] + 8) >> 4
        out[half::2, 1::2] = (3 * cs[:, 1:w + 1] + cs[:, 2:w + 2] + 7) >> 4
    return out.astype(np.uint8)


def _tables(oracle, Q, Qc):
    return (oracle.jpeg_Q() if Q is None else np.asarray(Q, np.float32),
            oracle.jpeg_Q_chroma() if Qc is None else np.asarray(Qc, np.float32))


def forward_rgb420(oracle, rgb, Q=None, Qc=None, keep=None):
    """(H, W, 3) u8 -> the (y, cb, cr) int16 zig-zag streams."""
    Q, Qc = _tables(oracle, Q, Qc)
    keep = oracle.ALL_COEFFS if keep is None else keep
    y, cb, cr = oracle.rgb_to_ycc(rgb)
    planes = (y, downsample_h2v2(cb), downsample_h2v2(cr))
    return tuple(oracle.zigzag_i16(oracle.dct(p.astype(np.float32), Q=Q if c == 0 else Qc, keep=keep))
                 for c, p in enumerate(planes))


def decode_planes(oracle, streams, Q=None, Qc=None):
    """The three decoded u8 planes (Y full, Cb and Cr half resolution) of the streams, before upsampling."""
    Q, Qc = _tables(oracle, Q, Qc)
    return tuple(oracle.to_u8(oracle.idct(oracle.unzigzag_i16(s), Q=Q if c == 0 else Qc)) for c, s in enumerate(streams))


def inverse_rgb420(oracle, streams, Q=None, Qc=None):
    """The (y, cb, cr) streams -> (H, W, 3) u8."""
    y, cb, cr = decode_planes(oracle, streams, Q, Qc)
    return oracle.ycc_to_rgb(y, upsample_h2v2_fancy(cb), upsample_h2v2_fancy(cr))
