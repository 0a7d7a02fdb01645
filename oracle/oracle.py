"""ctypes wrapper over oracle/liboracle.so (the CPU restatement, oracle/dct_oracle.c).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / reference legs.  The product package never imports it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle.so")

ALL_COEFFS = (1 << 64) - 1


def build(force: bool = False) -> str:
    """Compile liboracle.so (gcc, seconds).  Safe to call repeatedly."""
    src = os.path.join(_HERE, "dct_oracle.c")
    if force or not os.path.exists(_LIB) or os.path.getmtime(_LIB) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE, "oracle"])
    return _LIB


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
        u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
        L.oracle_haweel_T.restype = C.POINTER(C.c_float)
        L.oracle_jpeg_Q.restype = C.POINTER(C.c_float)
        L.oracle_dct2_T.argtypes = [f32p]
        L.oracle_zigzag_mask.restype = C.c_uint64
        L.oracle_zigzag_mask.argtypes = [C.c_int]
        L.oracle_fill_rand.argtypes = [f32p, C.c_size_t, C.c_uint]
        L.oracle_fill_rand_u8.argtypes = [u8p, C.c_size_t, C.c_uint]
        L.oracle_convert_to_float.argtypes = [u8p, f32p, C.c_size_t]
        L.oracle_convert_to_u8.argtypes = [f32p, u8p, C.c_size_t]
        L.oracle_dct.argtypes = [f32p, C.c_int, C.c_int, f32p, f32p, C.c_uint64, f32p, C.c_void_p, C.c_int]
        L.oracle_idct.argtypes = [f32p, C.c_int, C.c_int, f32p, f32p, f32p, C.c_int]
        L.oracle_roundtrip.argtypes = [f32p, C.c_int, C.c_int, f32p, f32p, C.c_uint64, C.c_void_p, f32p, C.c_int]
        L.oracle_roundtrip_u8.argtypes = [u8p, C.c_int, C.c_int, f32p, f32p, C.c_uint64, C.c_void_p, u8p, C.c_int]
        L.oracle_metrics_u8.argtypes = [u8p, u8p, C.c_size_t, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.oracle_metrics_f32.argtypes = [f32p, f32p, C.c_size_t, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.oracle_fnv_coef.restype = C.c_uint64
        L.oracle_fnv_coef.argtypes = [f32p, C.c_size_t]
        L.oracle_fnv_u8.restype = C.c_uint64
        L.oracle_fnv_u8.argtypes = [u8p, C.c_size_t]
        L.oracle_time_roundtrip.restype = C.c_double
        L.oracle_time_roundtrip.argtypes = [f32p, C.c_int, C.c_int, f32p, C.c_int, C.c_int]
        L.oracle_max_threads.restype = C.c_int
        i16p = np.ctypeslib.ndpointer(np.int16, flags="C_CONTIGUOUS")
        L.oracle_zigzag_i16.argtypes = [f32p, C.c_int, C.c_int, i16p]
        L.oracle_unzigzag_i16.argtypes = [i16p, C.c_int, C.c_int, f32p]
        L.oracle_jpeg_Q_chroma.restype = C.POINTER(C.c_float)
        L.oracle_rgb_to_ycc.argtypes = [u8p, C.c_size_t, u8p, u8p, u8p]
        L.oracle_ycc_to_rgb.argtypes = [u8p, u8p, u8p, C.c_size_t, u8p]
        L.oracle_roundtrip_rgb.argtypes = [u8p, C.c_int, C.c_int, f32p, f32p, f32p, C.c_uint64, u8p, C.c_void_p, C.c_void_p, C.c_int]
        L.oracle_huffman_spec.argtypes = [C.c_int, C.c_int, u8p, u8p, C.POINTER(C.c_int)]
        L.oracle_huffman_lengths.argtypes = [C.c_int, C.c_int, u8p]
        L.oracle_coded_bits.restype = C.c_uint64
        L.oracle_coded_bits.argtypes = [i16p, C.c_size_t, C.c_int]
        _lib = L
    return _lib


def haweel_T() -> np.ndarray:
    return np.ctypeslib.as_array(lib().oracle_haweel_T(), shape=(64,)).copy()


def jpeg_Q() -> np.ndarray:
    return np.ctypeslib.as_array(lib().oracle_jpeg_Q(), shape=(64,)).copy()


def jpeg_Q_chroma() -> np.ndarray:
    """ITU-T T.81 Annex K.2 chrominance table."""
    return np.ctypeslib.as_array(lib().oracle_jpeg_Q_chroma(), shape=(64,)).copy()


def rgb_to_ycc(rgb: np.ndarray):
    """libjpeg's jccolor.c conversion: interleaved (H, W, 3) u8 -> three (H, W) u8 planes."""
    rgb = np.ascontiguousarray(rgb, np.uint8)
    H, W = rgb.shape[:2]
    y, cb, cr = (np.empty((H, W), np.uint8) for _ in range(3))
    lib().oracle_rgb_to_ycc(rgb.reshape(-1), H * W, y.reshape(-1), cb.reshape(-1), cr.reshape(-1))
    return y, cb, cr


def ycc_to_rgb(y, cb, cr) -> np.ndarray:
    """libjpeg's jdcolor.c conversion: three (H, W) u8 planes -> interleaved (H, W, 3) u8."""
    H, W = y.shape
    rgb = np.empty((H, W, 3), np.uint8)
    lib().oracle_ycc_to_rgb(np.ascontiguousarray(y).reshape(-1), np.ascontiguousarray(cb).reshape(-1),
                            np.ascontiguousarray(cr).reshape(-1), H * W, rgb.reshape(-1))
    return rgb


def roundtrip_rgb(rgb: np.ndarray, T=None, Q=None, Qc=None, keep: int = ALL_COEFFS, want_planes: bool = False,
                  want_coef: bool = False, threads: int = 1):
    """Interleaved RGB u8 -> YCbCr (libjpeg) -> per-plane reference round trip (Q for Y, Qc for
    Cb/Cr) -> RGB u8.  Optionally also the (3, H, W) u8 planes after the round trip and the
    (3, H, W) f32 coefficient planes."""
    rgb = np.ascontiguousarray(rgb, np.uint8)
    H, W = rgb.shape[:2]
    T, Q = _tq(T, Q)
    Qc = jpeg_Q_chroma() if Qc is None else np.ascontiguousarray(Qc, np.float32).reshape(64)
    out = np.empty_like(rgb)
    planes = np.empty((3, H, W), np.uint8) if want_planes else None
    coef = np.empty((3, H, W), np.float32) if want_coef else None
    lib().oracle_roundtrip_rgb(rgb.reshape(-1), H, W, T, Q, Qc, keep, out.reshape(-1),
                               planes.ctypes.data if want_planes else None, coef.ctypes.data if want_coef else None, threads)
    res = (out,)
    if want_planes:
        res += (planes,)
    if want_coef:
        res += (coef,)
    return res[0] if len(res) == 1 else res


def huffman_spec(which: int, table: int):
    """(BITS[16], HUFFVAL) of the Annex K.3 table as a DHT marker carries it; which 0 DC / 1 AC."""
    bits, vals, n = np.zeros(16, np.uint8), np.zeros(256, np.uint8), C.c_int()
    lib().oracle_huffman_spec(which, table, bits, vals, C.byref(n))
    return bits, vals[: n.value].copy()


def huffman_lengths(which: int, table: int) -> np.ndarray:
    out = np.zeros(256, np.uint8)
    lib().oracle_huffman_lengths(which, table, out)
    return out


CODED_OUT_OF_RANGE = 1 << 63


def coded_bits(stream: np.ndarray, table: int = 0) -> int:
    """Baseline-JPEG entropy-coded size in bits of one plane's zig-zag int16 stream (.., 64).  Symbols
    outside the baseline categories count 0 bits and set CODED_OUT_OF_RANGE (bit 63), as on the GPU."""
    stream = np.ascontiguousarray(stream, np.int16)
    return int(lib().oracle_coded_bits(stream.reshape(-1), stream.size // 64, table))


def compression_factor(coef: np.ndarray, table: int = 0) -> float:
    """8*H*W / coded_bits of a coefficient plane (README.md:62-69 'Compr. Factor', see dct_oracle.c)."""
    H, W = coef.shape
    bits = coded_bits(zigzag_i16(coef), table)
    if bits & CODED_OUT_OF_RANGE:
        raise ValueError("coefficients outside the baseline-JPEG categories: no coded size")
    return 8.0 * H * W / bits


def dct2_T() -> np.ndarray:
    t = np.empty(64, np.float32)
    lib().oracle_dct2_T(t)
    return t


def zigzag_mask(k: int) -> int:
    return int(lib().oracle_zigzag_mask(k))


def zigzag_i16(coef: np.ndarray) -> np.ndarray:
    """float coefficient plane (H, W) -> block-major int16 zig-zag stream (H/8, W/8, 64)."""
    coef = np.ascontiguousarray(coef, np.float32)
    H, W = coef.shape
    out = np.empty((H // 8, W // 8, 64), np.int16)
    lib().oracle_zigzag_i16(coef, H, W, out)
    return out


def unzigzag_i16(stream: np.ndarray) -> np.ndarray:
    stream = np.ascontiguousarray(stream, np.int16)
    H, W = stream.shape[0] * 8, stream.shape[1] * 8
    out = np.empty((H, W), np.float32)
    lib().oracle_unzigzag_i16(stream, H, W, out)
    return out


def rand_image(n_rows: int, n_cols: int, seed: int = 42) -> np.ndarray:
    """The reference benchmark's input (srand(seed); rand()%256), float32."""
    img = np.empty((n_rows, n_cols), np.float32)
    lib().oracle_fill_rand(img.reshape(-1), img.size, seed)
    return img


def rand_image_u8(n_rows: int, n_cols: int, seed: int = 42) -> np.ndarray:
    img = np.empty((n_rows, n_cols), np.uint8)
    lib().oracle_fill_rand_u8(img.reshape(-1), img.size, seed)
    return img


def _tq(T, Q):
    T = haweel_T() if T is None else np.ascontiguousarray(T, np.float32).reshape(64)
    Q = jpeg_Q() if Q is None else np.ascontiguousarray(Q, np.float32).reshape(64)
    return T, Q


def dct(img: np.ndarray, T=None, Q=None, keep: int = ALL_COEFFS, want_shifted: bool = False, threads: int = 1):
    img = np.ascontiguousarray(img, np.float32)
    H, W = img.shape
    T, Q = _tq(T, Q)
    coef = np.empty_like(img)
    shifted = np.empty_like(img) if want_shifted else None
    lib().oracle_dct(img, H, W, T, Q, keep, coef, shifted.ctypes.data if want_shifted else None, threads)
    return (coef, shifted) if want_shifted else coef


def idct(coef: np.ndarray, T=None, Q=None, threads: int = 1) -> np.ndarray:
    coef = np.ascontiguousarray(coef, np.float32)
    H, W = coef.shape
    T, Q = _tq(T, Q)
    out = np.empty_like(coef)
    lib().oracle_idct(coef, H, W, T, Q, out, threads)
    return out


def roundtrip(img: np.ndarray, T=None, Q=None, keep: int = ALL_COEFFS, want_coef: bool = False, threads: int = 1):
    T, Q = _tq(T, Q)
    H, W = img.shape
    coef = np.empty((H, W), np.float32) if want_coef else None
    cptr = coef.ctypes.data if want_coef else None
    if img.dtype == np.uint8:
        img = np.ascontiguousarray(img)
        out = np.empty_like(img)
        lib().oracle_roundtrip_u8(img, H, W, T, Q, keep, cptr, out, threads)
    else:
        img = np.ascontiguousarray(img, np.float32)
        out = np.empty_like(img)
        lib().oracle_roundtrip(img, H, W, T, Q, keep, cptr, out, threads)
    return (out, coef) if want_coef else out


def to_u8(x: np.ndarray) -> np.ndarray:
    x = np.ascontiguousarray(x, np.float32)
    out = np.empty(x.shape, np.uint8)
    lib().oracle_convert_to_u8(x.reshape(-1), out.reshape(-1), x.size)
    return out


def metrics(x: np.ndarray, y: np.ndarray):
    """(MSE, PEEN%) of y against the original x; u8 or f32 arrays."""
    mse, peen = C.c_double(), C.c_double()
    if x.dtype == np.uint8:
        lib().oracle_metrics_u8(np.ascontiguousarray(x).reshape(-1), np.ascontiguousarray(y).reshape(-1), x.size, mse, peen)
    else:
        lib().oracle_metrics_f32(np.ascontiguousarray(x, np.float32).reshape(-1),
                                 np.ascontiguousarray(y, np.float32).reshape(-1), x.size, mse, peen)
    return mse.value, peen.value


def fnv_coef(coef: np.ndarray) -> int:
    return int(lib().oracle_fnv_coef(np.ascontiguousarray(coef, np.float32).reshape(-1), coef.size))


def fnv_u8(p: np.ndarray) -> int:
    return int(lib().oracle_fnv_u8(np.ascontiguousarray(p, np.uint8).reshape(-1), p.size))


def time_roundtrip(img: np.ndarray, reps: int = 3, threads: int = 1) -> float:
    """Best-of-reps wall seconds for one fused DCT->quant->IDCT pass over img (f32)."""
    img = np.ascontiguousarray(img, np.float32)
    out = np.empty_like(img)
    return float(lib().oracle_time_roundtrip(img, img.shape[0], img.shape[1], out, reps, threads))


def max_threads() -> int:
    return int(lib().oracle_max_threads())
