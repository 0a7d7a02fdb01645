"""ctypes host side over the C ABI (include/b200dct.h) and the compat library.

Tensors are torch CUDA tensors (torch is used only for device memory and streams) for the
device entry points, numpy arrays for the host-buffer round trip.  The functions named
like the reference's (``dct_all_blocks_cuda`` ...) keep its argument order
``(image, H, W, T, result)`` -- height before width (main_newAppr.cu:23-24) -- and its side
effects, by calling the same compiled wrappers a C++ caller would link.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ALL_COEFFS = (1 << 64) - 1

F32, U8, I16, I16_ZIGZAG = 0, 1, 2, 3
PATH_AUTO, PATH_DIRECT, PATH_TMA = 0, 1, 2
INVERSE_AUTO, INVERSE_EXACT, INVERSE_FACTORED = 0, 1, 2
DENSE_AUTO, DENSE_CHAIN, DENSE_SYMMETRIC, DENSE_MMA = 0, 1, 2, 3


class B200DCTError(RuntimeError):
    pass


def lib_path(name: str = "libb200dct.so") -> str:
    # B200DCT_LIB_DIR: developer override used to A/B experimental builds of the library
    return os.path.join(os.environ.get("B200DCT_LIB_DIR", _HERE), name)


_lib = None
_compat = None


def lib() -> C.CDLL:
    """Load libb200dct.so.  Fails loudly if it has not been built: there is no fallback."""
    global _lib
    if _lib is None:
        p = lib_path()
        if not os.path.exists(p):
            raise B200DCTError(
                f"{p} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
        L = C.CDLL(p)
        vp, sz, i, u64 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint64
        L.b200dct_plan_create.argtypes = [C.POINTER(vp)]
        L.b200dct_plan_destroy.argtypes = [vp]
        L.b200dct_plan_destroy.restype = None
        L.b200dct_plan_set_quant.argtypes = [vp, C.POINTER(C.c_float)]
        L.b200dct_plan_get_quant.argtypes = [vp, C.POINTER(C.c_float)]
        L.b200dct_plan_set_transform.argtypes = [vp, C.POINTER(C.c_float)]
        L.b200dct_plan_set_transform_device.argtypes = [vp, vp]
        L.b200dct_plan_set_keep_mask.argtypes = [vp, u64]
        L.b200dct_zigzag_mask.argtypes = [i]
        L.b200dct_zigzag_mask.restype = u64
        L.b200dct_plan_set_path.argtypes = [vp, i]
        L.b200dct_plan_is_sparse.argtypes = [vp]
        L.b200dct_plan_set_inverse.argtypes = [vp, i]
        L.b200dct_plan_set_dense.argtypes = [vp, i]
        L.b200dct_plan_kernel_kind.argtypes = [vp]
        L.b200dct_forward.argtypes = [vp, vp, i, sz, vp, i, sz, vp, i, i, vp]
        L.b200dct_inverse.argtypes = [vp, vp, i, sz, vp, i, sz, i, i, vp]
        L.b200dct_roundtrip.argtypes = [vp, vp, i, sz, vp, i, sz, vp, i, sz, i, i, vp]
        L.b200dct_metrics_workspace_bytes.argtypes = [i, i]
        L.b200dct_metrics_workspace_bytes.restype = sz
        L.b200dct_roundtrip_metrics.argtypes = [vp, vp, i, sz, vp, i, sz, vp, i, sz, i, i, vp, vp, sz, vp]
        L.b200dct_roundtrip_any.argtypes = [vp, vp, i, sz, vp, sz, i, i, vp]
        L.b200dct_roundtrip_batch.argtypes = [vp, i, C.POINTER(vp), C.POINTER(vp), i, sz, sz, i, i, vp]
        L.b200dct_roundtrip_host.argtypes = [vp, vp, i, vp, i, i, i]
        L.b200dct_plan_set_chroma_quant.argtypes = [vp, C.POINTER(C.c_float)]
        L.b200dct_plan_get_chroma_quant.argtypes = [vp, C.POINTER(C.c_float)]
        L.b200dct_roundtrip_rgb.argtypes = [vp, vp, sz, vp, sz, vp, sz, i, i, vp]
        L.b200dct_forward_rgb.argtypes = [vp, vp, sz, vp, sz, i, i, vp]
        L.b200dct_inverse_rgb.argtypes = [vp, vp, sz, vp, sz, i, i, vp]
        L.b200dct_zigzag_coded_bits.argtypes = [vp, sz, i, i, i, vp, vp]
        L.b200dct_host_pipeline_create.argtypes = [C.POINTER(vp), sz, i]
        L.b200dct_host_pipeline_destroy.argtypes = [vp]
        L.b200dct_host_pipeline_destroy.restype = None
        L.b200dct_host_pipeline_chunk_bytes.argtypes = [vp]
        L.b200dct_host_pipeline_chunk_bytes.restype = sz
        L.b200dct_host_pipeline_submit.argtypes = [vp, vp, vp, i, vp, i, i, i, C.POINTER(C.c_ulonglong)]
        L.b200dct_host_pipeline_wait.argtypes = [vp, C.c_ulonglong]
        L.b200dct_host_pipeline_drain.argtypes = [vp]
        L.b200dct_host_pipeline_last_launch_count.argtypes = [vp]
        L.b200dct_metrics_accumulate.argtypes = [vp, vp, i, sz, i, i, vp, vp]
        L.b200dct_time_calls.argtypes = [vp, i, vp, i, sz, vp, i, sz, vp, i, sz, i, i, i, C.POINTER(C.c_float), vp]
        L.b200dct_selftest_division.argtypes = [C.c_float, C.c_ulonglong, C.c_ulonglong, vp, vp]
        L.b200dct_last_launch_count.restype = i
        L.b200dct_last_path.restype = C.c_char_p
        L.b200dct_error_string.argtypes = [i]
        L.b200dct_error_string.restype = C.c_char_p
        _lib = L
    return _lib


def compat_lib() -> C.CDLL:
    global _compat
    if _compat is None:
        lib()  # dependency, and the loud failure
        L = C.CDLL(lib_path("libb200dct_compat.so"))
        vp, i = C.c_void_p, C.c_int
        L.b200dct_compat_set_quant.argtypes = [C.POINTER(C.c_float)]
        L.b200dct_compat_set_keep_mask.argtypes = [C.c_uint64]
        L.b200dct_compat_set_options.argtypes = [i, i]
        L.b200dct_compat_set_options.restype = None
        L.b200dct_compat_cache_transform.argtypes = [i]
        L.b200dct_compat_cache_transform.restype = None
        L.b200dct_compat_last_ms.restype = C.c_float
        for f in (L.b200dct_compat_dct, L.b200dct_compat_idct, L.b200dct_compat_idct_inplace_dequant):
            f.argtypes = [vp, i, i, vp, vp]
            f.restype = None
        _compat = L
    return _compat


def _check(rc: int) -> None:
    if rc != 0:
        raise B200DCTError(f"b200dct error {rc}: {lib().b200dct_error_string(rc).decode()}")


def zigzag_mask(k: int) -> int:
    return int(lib().b200dct_zigzag_mask(int(k)))


def _f64(a) -> "C.Array":
    a = np.ascontiguousarray(a, np.float32).reshape(64)
    return (C.c_float * 64)(*a.tolist())


class Plan:
    """T, Q and the retained-coefficient mask (b200dct_plan)."""

    def __init__(self, T=None, Q=None, keep: int = ALL_COEFFS, path: int = PATH_AUTO, inverse: int = INVERSE_AUTO,
                 dense: int = DENSE_AUTO, Qc=None):
        self._h = C.c_void_p()
        _check(lib().b200dct_plan_create(C.byref(self._h)))
        if T is not None:
            self.set_transform(T)
        if Q is not None:
            self.set_quant(Q)
        if Qc is not None:
            self.set_chroma_quant(Qc)
        if keep != ALL_COEFFS:
            self.set_keep_mask(keep)
        if path != PATH_AUTO:
            self.set_path(path)
        if inverse != INVERSE_AUTO:
            self.set_inverse(inverse)
        if dense != DENSE_AUTO:
            self.set_dense(dense)

    def set_transform(self, T) -> None:
        _check(lib().b200dct_plan_set_transform(self._h, _f64(T)))

    def set_quant(self, Q) -> None:
        _check(lib().b200dct_plan_set_quant(self._h, _f64(Q)))

    def quant(self) -> np.ndarray:
        q = (C.c_float * 64)()
        _check(lib().b200dct_plan_get_quant(self._h, q))
        return np.array(q[:], np.float32)

    def set_chroma_quant(self, Q) -> None:
        """Quantisation table of the Cb / Cr planes of roundtrip_rgb (default: T.81 Annex K.2)."""
        _check(lib().b200dct_plan_set_chroma_quant(self._h, _f64(Q)))

    def chroma_quant(self) -> np.ndarray:
        q = (C.c_float * 64)()
        _check(lib().b200dct_plan_get_chroma_quant(self._h, q))
        return np.array(q[:], np.float32)

    def set_keep_mask(self, mask: int) -> None:
        _check(lib().b200dct_plan_set_keep_mask(self._h, mask & ALL_COEFFS))

    def set_path(self, path: int) -> None:
        _check(lib().b200dct_plan_set_path(self._h, path))

    def set_inverse(self, mode: int) -> None:
        """INVERSE_EXACT: the reference's FMA chains everywhere (u8 pixels bit-identical to the
        reference); INVERSE_AUTO / INVERSE_FACTORED: butterfly inverse for 8-bit output (+-1 LSB)."""
        _check(lib().b200dct_plan_set_inverse(self._h, mode))

    def set_dense(self, mode: int) -> None:
        """DENSE_CHAIN: ordered FMA chains for a dense T (bit-identical to the reference's chain order with that T);
        DENSE_AUTO / DENSE_SYMMETRIC: even/odd evaluation when T has the DCT-II symmetry;
        DENSE_MMA: the tensor-core arm (f32 fused round trips on mma.sync TF32 with hi/lo splits), opt-in."""
        _check(lib().b200dct_plan_set_dense(self._h, mode))

    @property
    def kernel_kind(self) -> int:
        """0 ordered chains (dense T), 1 Haweel sparse kernels, 2 symmetric dense kernels."""
        return int(lib().b200dct_plan_kernel_kind(self._h))

    @property
    def is_sparse(self) -> bool:
        return bool(lib().b200dct_plan_is_sparse(self._h))

    def __del__(self):
        try:
            if self._h and _lib is not None:
                _lib.b200dct_plan_destroy(self._h)
                self._h = None
        except Exception:
            pass


_default_plan = None


def _plan(plan):
    global _default_plan
    if plan is not None:
        return plan
    if _default_plan is None:
        _default_plan = Plan()
    return _default_plan


def _dt(t) -> int:
    import torch

    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.uint8:
        return U8
    if t.dtype == torch.int16:
        return I16
    raise B200DCTError(f"unsupported dtype {t.dtype}")


def _plane(t):
    """(ptr, dtype code, pitch bytes, H, W) of a 2-d (or batch-as-rows 3-d) CUDA tensor."""
    if not t.is_cuda:
        raise B200DCTError("device entry points take CUDA tensors (no CPU path)")
    if t.dim() == 3:  # B x H x W stored back to back == one (B*H) x W image
        if not t.is_contiguous():
            raise B200DCTError("batched tensors must be contiguous")
        if t.shape[-2] % 8:
            raise B200DCTError("batched images need a height that is a multiple of 8 (blocks must not straddle images)")
        t = t.view(-1, t.shape[-1])
    if t.dim() != 2 or t.stride(1) != 1:
        raise B200DCTError("expected a row-major 2-d tensor")
    return t.data_ptr(), _dt(t), t.stride(0) * t.element_size(), t.shape[0], t.shape[1]


def _same_plane(t, H, W, what, dtypes=None):
    """_plane(t) for a tensor that must describe the same H x W image: the C side trusts H, W and
    the pitch, so a smaller or differently shaped tensor would mean out-of-bounds device writes."""
    p, dt, pitch, h, w = _plane(t)
    if (h, w) != (H, W):
        raise B200DCTError(f"{what}: shape {tuple(t.shape)} does not describe the {H}x{W} image of the call")
    if dtypes is not None and t.dtype not in dtypes:
        raise B200DCTError(f"{what}: dtype {t.dtype} not allowed here")
    return p, dt, pitch


def _zz_same(t, H, W, what):
    p, dt, pitch, h, w = _zz_plane(t)
    if (h, w) != (H, W):
        raise B200DCTError(f"{what}: stream shape {tuple(t.shape)} does not match the {H}x{W} image")
    return p, dt, pitch


def _zz_plane(t):
    """(ptr, dtype code, pitch bytes, H, W) of a zig-zag coefficient stream: an int16 CUDA tensor of
    shape (H/8, W/8, 64) -- block-major, 64 coefficients per block in JPEG zig-zag order."""
    import torch

    if not (t.is_cuda and t.dtype == torch.int16 and t.dim() == 3 and t.shape[2] == 64
            and t.stride(2) == 1 and t.stride(1) == 64):
        raise B200DCTError("zig-zag streams are int16 CUDA tensors of shape (H/8, W/8, 64)")
    return t.data_ptr(), I16_ZIGZAG, t.stride(0) * 2, t.shape[0] * 8, t.shape[1] * 8


def empty_zigzag(H: int, W: int, device):
    import torch

    return torch.empty((H // 8, W // 8, 64), dtype=torch.int16, device=device)


def _stream(stream):
    import torch

    s = torch.cuda.current_stream() if stream is None else stream
    return C.c_void_p(s.cuda_stream)


class _on:
    """Scope of one call: the tensor's device and the caller's stream are made current, so that
    every allocation, launch and read-back of the call is ordered on ONE stream (torch's caching
    allocator ties a block to the stream that was current when it was allocated)."""

    def __init__(self, t, stream):
        import torch

        # the common case -- the tensor lives on the current device, the call runs on the current stream --
        # needs no context switch at all (two context managers cost ~4 us per call, more than a 256^2 kernel)
        self._dev = None if t.device.index == torch.cuda.current_device() else torch.cuda.device(t.device)
        self._st = torch.cuda.stream(stream) if stream is not None and stream != torch.cuda.current_stream(t.device) else None

    def __enter__(self):
        if self._dev is not None:
            self._dev.__enter__()
        if self._st is not None:
            self._st.__enter__()
        return self

    def __exit__(self, *a):
        if self._st is not None:
            self._st.__exit__(*a)
        if self._dev is not None:
            return self._dev.__exit__(*a)
        return False


def forward(img, coef=None, plan: Plan | None = None, coef_dtype=None, shifted=None, stream=None, zigzag=False):
    """coef = round(T.(img-128).T^T / Q); img f32|u8 CUDA tensor; coef f32 (default) or int16 plane,
    or (zigzag=True) the block-major int16 zig-zag stream of shape (H/8, W/8, 64)."""
    import torch

    ip, idt, ipitch, H, W = _plane(img)
    with _on(img, stream):
        if coef is None:
            coef = empty_zigzag(H, W, img.device) if zigzag else torch.empty(img.shape, dtype=coef_dtype or torch.float32, device=img.device)
        cp, cdt, cpitch = _zz_same(coef, H, W, "coef") if zigzag else _same_plane(coef, H, W, "coef", (torch.float32, torch.int16))
        sp = None
        if shifted is not None:
            # the C side writes img-128 as f32 with the INPUT's pitch (b200dct_forward)
            sp, _, spitch = _same_plane(shifted, H, W, "shifted", (torch.float32,))
            if img.dtype != torch.float32 or spitch != ipitch:
                raise B200DCTError("shifted: needs a float32 image and a float32 buffer with the image's row pitch")
        _check(lib().b200dct_forward(_plan(plan)._h, ip, idt, ipitch, cp, cdt, cpitch, sp, H, W, _stream(stream)))
    return coef


def inverse(coef, img=None, plan: Plan | None = None, img_dtype=None, stream=None, zigzag=False):
    """img = T^T.(coef*Q).T + 128; coef f32|int16 plane or (zigzag=True) the zig-zag stream;
    img f32 (unclamped) or u8 (clamp+truncate)."""
    import torch

    cp, cdt, cpitch, H, W = _zz_plane(coef) if zigzag else _plane(coef)
    with _on(coef, stream):
        if img is None:
            img = torch.empty((H, W) if zigzag else coef.shape, dtype=img_dtype or torch.float32, device=coef.device)
        ip, idt, ipitch = _same_plane(img, H, W, "img", (torch.float32, torch.uint8))
        _check(lib().b200dct_inverse(_plan(plan)._h, cp, cdt, cpitch, ip, idt, ipitch, H, W, _stream(stream)))
    return img


def roundtrip(img, out=None, coef=None, plan: Plan | None = None, stream=None, zigzag=False):
    """Fused DCT -> quantise -> dequantise -> IDCT in one pass; optional coefficient plane
    (zigzag=True: `coef` is the block-major int16 zig-zag stream)."""
    import torch

    ip, idt, ipitch, H, W = _plane(img)
    with _on(img, stream):
        if out is None:
            out = torch.empty_like(img)
        op, odt, opitch = _same_plane(out, H, W, "out", (img.dtype,))
        if coef is not None:
            cp, cdt, cpitch = _zz_same(coef, H, W, "coef") if zigzag else _same_plane(coef, H, W, "coef", (torch.float32, torch.int16))
        else:
            cp, cdt, cpitch = None, F32, 0
        _check(lib().b200dct_roundtrip(_plan(plan)._h, ip, idt, ipitch, op, odt, opitch, cp, cdt, cpitch, H, W,
                                       _stream(stream)))
    return out


def roundtrip_any(img, out=None, plan: Plan | None = None, stream=None):
    """Round trip of a 2-d CUDA tensor of ANY height/width/alignment: aligned multiples of 8 take
    the fast path, anything else one pass of the edge-replicating kernel (no scratch image);
    `out` may be `img` itself or a view inside a larger tensor."""
    import torch

    if not (img.is_cuda and img.dim() == 2 and img.stride(1) == 1):
        raise B200DCTError("expected a row-major 2-d CUDA tensor")
    with _on(img, stream):
        if out is None:
            out = torch.empty_like(img)
        if not out.is_cuda or out.shape != img.shape or out.dtype != img.dtype or out.stride(1) != 1:
            raise B200DCTError("out must match img")
        _check(lib().b200dct_roundtrip_any(_plan(plan)._h, img.data_ptr(), _dt(img), img.stride(0) * img.element_size(),
                                           out.data_ptr(), out.stride(0) * out.element_size(), img.shape[0], img.shape[1],
                                           _stream(stream)))
    return out


class ImageBatch:
    """A list of separately allocated CUDA images of ONE shape, dtype (float32 or uint8) and row pitch
    with their outputs, validated once: `run()` is then a single call of b200dct_roundtrip_batch (one
    launch per 64 images).  `outs`: matching list (entries may be the inputs themselves), allocated
    when omitted.  The batch keeps its tensors alive."""

    def __init__(self, imgs, outs=None):
        import torch

        self.imgs = list(imgs)
        if not self.imgs:
            raise B200DCTError("an image batch needs at least one image")
        first = self.imgs[0]
        _, self._dt, self._ipitch, self.H, self.W = _plane(first)
        with torch.cuda.device(first.device):
            self.outs = [torch.empty_like(t) for t in self.imgs] if outs is None else list(outs)
        if len(self.outs) != len(self.imgs):
            raise B200DCTError("outs must have one entry per image")
        n = len(self.imgs)
        self._in, self._out = (C.c_void_p * n)(), (C.c_void_p * n)()
        self._opitch = None
        for k, (a, b) in enumerate(zip(self.imgs, self.outs)):
            if a.dim() != 2 or b.dim() != 2 or a.device != first.device or b.device != first.device:
                raise B200DCTError("a batch is a list of 2-d images on one device")
            p, d, pitch, h, w = _plane(a)
            if (d, pitch, h, w) != (self._dt, self._ipitch, self.H, self.W):
                raise B200DCTError(f"image {k}: every image of a batch has the shape, dtype and pitch of the first")
            q, _, qpitch = _same_plane(b, self.H, self.W, f"outs[{k}]", (a.dtype,))
            if self._opitch is None:
                self._opitch = qpitch
            if qpitch != self._opitch:
                raise B200DCTError(f"outs[{k}]: every output of a batch has the pitch of the first")
            self._in[k], self._out[k] = p, q

    def __len__(self):
        return len(self.imgs)

    def run(self, plan: Plan | None = None, stream=None):
        with _on(self.imgs[0], stream):
            _check(lib().b200dct_roundtrip_batch(_plan(plan)._h, len(self.imgs), self._in, self._out, self._dt,
                                                 self._ipitch, self._opitch, self.H, self.W, _stream(stream)))
        return self.outs


def roundtrip_batch(imgs, outs=None, plan: Plan | None = None, stream=None):
    """Fused round trip of a list of separately allocated CUDA images of one shape, dtype and pitch in one
    launch per 64 images: the results are those of `roundtrip` on every image, bit for bit.  For a batch
    that is processed repeatedly build an `ImageBatch` once and call its `run()`."""
    imgs = list(imgs)
    if not imgs:
        return []
    import torch

    with _on(imgs[0], stream):      # allocation of missing outputs on the caller's stream
        batch = ImageBatch(imgs, [torch.empty_like(t) for t in imgs] if outs is None else outs)
    return batch.run(plan, stream)


def _rgb_image(t, H, W, what):
    """An interleaved (H, W, 3) uint8 CUDA tensor with rows of its own pitch (H, W None: any size)."""
    import torch

    if not (t.is_cuda and t.dtype == torch.uint8 and t.dim() == 3 and t.shape[2] == 3 and t.stride(2) == 1 and t.stride(1) == 3
            and (H is None or tuple(t.shape) == (H, W, 3))):
        raise B200DCTError("expected an interleaved (H, W, 3) uint8 CUDA tensor" if H is None else
                           f"{what} must be an interleaved (H, W, 3) uint8 CUDA tensor like rgb")


def _rgb_streams(t, H, W):
    """(pointer, plane stride in bytes) of the (3, H/8, W/8, 64) int16 zig-zag streams of Y, Cb, Cr."""
    import torch

    if not (t.is_cuda and t.dtype == torch.int16 and t.dim() == 4 and (H is None or tuple(t.shape) == (3, H // 8, W // 8, 64))
            and t.shape[0] == 3 and t.shape[3] == 64 and t[0].is_contiguous()):
        raise B200DCTError("streams must be a (3, H/8, W/8, 64) int16 CUDA tensor")
    return t.data_ptr(), t.stride(0) * 2


def roundtrip_rgb(rgb, out=None, streams=None, plan: Plan | None = None, stream=None):
    """Colour round trip in one pass (b200dct_roundtrip_rgb): `rgb` is an (H, W, 3) uint8 CUDA
    tensor (interleaved, as the reference's loader returns colour files); RGB -> YCbCr (libjpeg)
    -> per-plane DCT / quantise (luminance table for Y, chrominance table for Cb, Cr) / IDCT ->
    RGB.  `streams`: optional (3, H/8, W/8, 64) int16 tensor receiving the zig-zag coefficient
    streams of Y, Cb, Cr."""
    import torch

    _rgb_image(rgb, None, None, "rgb")
    H, W = int(rgb.shape[0]), int(rgb.shape[1])
    with _on(rgb, stream):
        if out is None:
            out = torch.empty_like(rgb)
        _rgb_image(out, H, W, "out")
        zp, zplane = _rgb_streams(streams, H, W) if streams is not None else (None, 0)
        _check(lib().b200dct_roundtrip_rgb(_plan(plan)._h, rgb.data_ptr(), rgb.stride(0), out.data_ptr(), out.stride(0),
                                           zp, zplane, H, W, _stream(stream)))
    return out


def forward_rgb(rgb, streams=None, plan: Plan | None = None, stream=None):
    """First half of `roundtrip_rgb` (b200dct_forward_rgb): an (H, W, 3) uint8 CUDA tensor -> YCbCr ->
    per-plane DCT / quantise -> the (3, H/8, W/8, 64) int16 zig-zag coefficient streams of Y, Cb, Cr
    (written into `streams` when given).  They are what `roundtrip_rgb(rgb, streams=...)` writes."""
    import torch

    _rgb_image(rgb, None, None, "rgb")
    H, W = int(rgb.shape[0]), int(rgb.shape[1])
    with _on(rgb, stream):
        if streams is None:
            streams = torch.empty((3, H // 8, W // 8, 64), dtype=torch.int16, device=rgb.device)
        zp, zplane = _rgb_streams(streams, H, W)
        _check(lib().b200dct_forward_rgb(_plan(plan)._h, rgb.data_ptr(), rgb.stride(0), zp, zplane, H, W, _stream(stream)))
    return streams


def inverse_rgb(streams, out=None, plan: Plan | None = None, stream=None):
    """Second half of `roundtrip_rgb` (b200dct_inverse_rgb): the (3, H/8, W/8, 64) int16 zig-zag streams
    of Y, Cb, Cr -> per-plane dequantise / IDCT -> RGB, an (H, W, 3) uint8 CUDA tensor (written into
    `out` when given).  inverse_rgb(forward_rgb(x)) == roundtrip_rgb(x) bit for bit with the same plan."""
    import torch

    zp, zplane = _rgb_streams(streams, None, None)
    H, W = int(streams.shape[1]) * 8, int(streams.shape[2]) * 8
    with _on(streams, stream):
        if out is None:
            out = torch.empty((H, W, 3), dtype=torch.uint8, device=streams.device)
        _rgb_image(out, H, W, "out")
        _check(lib().b200dct_inverse_rgb(_plan(plan)._h, zp, zplane, out.data_ptr(), out.stride(0), H, W, _stream(stream)))
    return out


def coded_bits(zz, table: int = 0, stream=None) -> int:
    """Baseline-JPEG entropy-coded size in bits of one plane's zig-zag stream, an (H/8, W/8, 64)
    int16 CUDA tensor (b200dct_zigzag_coded_bits); table 0 = luminance codes, 1 = chrominance."""
    import torch

    p, _, pitch, H, W = _zz_plane(zz)
    with _on(zz, stream):
        acc = torch.zeros(1, dtype=torch.int64, device=zz.device)
        _check(lib().b200dct_zigzag_coded_bits(p, pitch, H, W, int(table), acc.data_ptr(), _stream(stream)))
        return int(acc.item())


def compression_factor(zz, table: int = 0, stream=None) -> float:
    """8*H*W / coded_bits: the README's 'Compr. Factor' (README.md:62-69) under the baseline-JPEG
    entropy coder.  `zz`: one plane's stream, or a (3, ...) stack (Y with the luminance codes,
    Cb and Cr with the chrominance codes; CF of the whole colour image)."""
    if zz.dim() == 4:
        bits = sum(coded_bits(zz[c], 0 if c == 0 else 1, stream) for c in range(zz.shape[0]))
        return 8.0 * zz.shape[0] * zz.shape[1] * zz.shape[2] * 64 / bits
    return 8.0 * zz.shape[0] * zz.shape[1] * 64 / coded_bits(zz, table, stream)


def roundtrip_with_metrics(img, out=None, coef=None, plan: Plan | None = None, stream=None, zigzag=False):
    """Fused round trip that also returns (MSE, PEEN%, non-zero coefficient count) of the
    pass, computed inside the kernel (b200dct_roundtrip_metrics).  zigzag=True: `coef` is the
    block-major int16 zig-zag stream."""
    import torch

    ip, idt, ipitch, H, W = _plane(img)
    with _on(img, stream):     # workspace, zero-fill, kernels and the read-back all on the caller's stream
        if out is None:
            out = torch.empty_like(img)
        op, odt, opitch = _same_plane(out, H, W, "out", (img.dtype,))
        if coef is None:
            cp, cdt, cpitch = None, F32, 0
        else:
            cp, cdt, cpitch = _zz_same(coef, H, W, "coef") if zigzag else _same_plane(coef, H, W, "coef", (torch.float32, torch.int16))
        nbytes = int(lib().b200dct_metrics_workspace_bytes(H, W))
        ws = torch.empty(max(1, nbytes // 8), dtype=torch.float64, device=img.device)
        acc = torch.zeros(3, dtype=torch.float64, device=img.device)
        _check(lib().b200dct_roundtrip_metrics(_plan(plan)._h, ip, idt, ipitch, op, odt, opitch, cp, cdt, cpitch, H, W,
                                               acc.data_ptr(), ws.data_ptr(), nbytes, _stream(stream)))
        sse, energy, nnz = acc.tolist()
    n = H * W
    return out, (sse / n, 100.0 * (sse / energy) ** 0.5 if energy > 0 else 0.0, int(nnz))


def _hostptr(a):
    """(pointer, dtype code, shape) of a contiguous numpy array or CPU torch tensor."""
    import torch

    if isinstance(a, np.ndarray):
        if not a.flags.c_contiguous:
            raise B200DCTError("host arrays must be C-contiguous")
        dt = {np.dtype(np.float32): F32, np.dtype(np.uint8): U8}.get(a.dtype)
        if dt is None:
            raise B200DCTError("host round trips take float32 or uint8 pixels")
        return a.ctypes.data, dt, tuple(a.shape)
    if isinstance(a, torch.Tensor) and not a.is_cuda and a.is_contiguous():
        dt = _dt(a)
        if dt == I16:
            raise B200DCTError("host round trips take float32 or uint8 pixels")
        return a.data_ptr(), dt, tuple(a.shape)
    raise B200DCTError("expected a contiguous numpy array or CPU torch tensor")


def roundtrip_host(h_in, h_out=None, plan: Plan | None = None):
    """Host buffers in, host buffers out (numpy arrays or pinned CPU torch tensors):
    chunked H2D -> fused kernel -> D2H pipeline inside the library.  Synchronous."""
    import torch

    ip, idt, shape = _hostptr(h_in)
    if h_out is None:
        h_out = np.empty_like(h_in) if isinstance(h_in, np.ndarray) else torch.empty_like(h_in)
    op, odt, oshape = _hostptr(h_out)
    if oshape != shape or len(shape) < 2:
        raise B200DCTError("shape mismatch")
    H = int(np.prod(shape[:-1]))
    _check(lib().b200dct_roundtrip_host(_plan(plan)._h, ip, idt, op, odt, H, int(shape[-1])))
    return h_out


class HostPipeline:
    """A sequence of host-buffer round trips whose images overlap (b200dct_host_pipeline_*):
    `submit` only enqueues; `wait(ticket)` / `drain()` (or leaving the `with` block) completes.
    Buffers must be pinned for the copies to be asynchronous and must stay alive (and `h_out`
    unread) until waited for."""

    def __init__(self, plan: Plan | None = None, chunk_bytes: int = 0, slots: int = 0):
        self._plan = _plan(plan)
        self._h = C.c_void_p()
        self._keep = {}
        _check(lib().b200dct_host_pipeline_create(C.byref(self._h), int(chunk_bytes), int(slots)))

    @property
    def chunk_bytes(self) -> int:
        return int(lib().b200dct_host_pipeline_chunk_bytes(self._h))

    def submit(self, h_in, h_out, plan: Plan | None = None) -> int:
        ip, idt, shape = _hostptr(h_in)
        op, odt, oshape = _hostptr(h_out)
        if oshape != shape or len(shape) < 2:
            raise B200DCTError("shape mismatch")
        t = C.c_ulonglong()
        H = int(np.prod(shape[:-1]))
        _check(lib().b200dct_host_pipeline_submit(self._h, (plan or self._plan)._h, ip, idt, op, odt, H, int(shape[-1]), C.byref(t)))
        self._keep[t.value] = (h_in, h_out)      # the library reads/writes them until the ticket completes
        return int(t.value)

    def wait(self, ticket: int) -> None:
        _check(lib().b200dct_host_pipeline_wait(self._h, int(ticket)))
        for k in [k for k in self._keep if k <= ticket]:
            del self._keep[k]

    def drain(self) -> None:
        _check(lib().b200dct_host_pipeline_drain(self._h))
        self._keep.clear()

    def last_launch_count(self) -> int:
        return int(lib().b200dct_host_pipeline_last_launch_count(self._h))

    def close(self) -> None:
        if self._h:
            lib().b200dct_host_pipeline_destroy(self._h)
            self._h = C.c_void_p()
            self._keep.clear()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        try:
            if a[0] is None:
                self.drain()
        finally:
            self.close()

    def __del__(self):
        try:
            if _lib is not None:
                self.close()
        except Exception:
            pass


def metrics(ref_img, test_img, stream=None):
    """(MSE, PEEN%) of test_img against ref_img, accumulated on the device in double."""
    import torch

    rp, rdt, rpitch, H, W = _plane(ref_img)
    tp, tdt, tpitch = _same_plane(test_img, H, W, "test_img", (ref_img.dtype,))
    if rdt != tdt or rpitch != tpitch or rdt not in (F32, U8):
        raise B200DCTError("metrics needs two float32 or uint8 images of the same dtype and pitch")
    with _on(ref_img, stream):
        acc = torch.zeros(2, dtype=torch.float64, device=ref_img.device)
        _check(lib().b200dct_metrics_accumulate(rp, tp, rdt, rpitch, H, W, acc.data_ptr(), _stream(stream)))
        sse, energy = acc.tolist()
    n = H * W
    return sse / n, (100.0 * (sse / energy) ** 0.5 if energy > 0 else 0.0)


def time_calls(which: str, a, b, c=None, plan: Plan | None = None, iters: int = 100, stream=None) -> float:
    """Average device ms of `iters` back-to-back calls issued from C (b200dct_time_calls).
    which: "roundtrip" (a -> b [, c = coefficient plane]), "forward", "inverse", or
    "split" (forward a -> c, inverse c -> b)."""
    import torch

    code = {"roundtrip": 0, "forward": 1, "inverse": 2, "split": 3}[which]
    ap, adt, apitch, H, W = _plane(a)
    bp, bdt, bpitch = _same_plane(b, H, W, "b")
    cp, cdt, cpitch = (None, F32, 0) if c is None else _same_plane(c, H, W, "c")
    ms = C.c_float()
    with torch.cuda.device(a.device):
        _check(lib().b200dct_time_calls(_plan(plan)._h, code, ap, adt, apitch, bp, bdt, bpitch, cp, cdt, cpitch,
                                        H, W, int(iters), C.byref(ms), _stream(stream)))
    return float(ms.value)


def last_launch_count() -> int:
    return int(lib().b200dct_last_launch_count())


def last_path() -> str:
    return lib().b200dct_last_path().decode()


# ---------------------------------------------------------------- reference-named entry points
def _compat_call(fn, a, H, W, T, result):
    import torch

    for t in (a, T, result):
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise B200DCTError("the reference's entry points take contiguous float32 device buffers")
    if a.numel() < H * W or result.numel() < H * W or T.numel() < 64:
        raise B200DCTError("buffer smaller than H*W")
    # the compiled wrappers keep the reference's contract (print and exit(EXIT_FAILURE) on error,
    # main_newAppr.cu:9-17): catch here what would otherwise end the interpreter
    if H <= 0 or W <= 0 or H % 8 or W % 8:
        raise B200DCTError("the reference's entry points need H and W to be positive multiples of 8")
    if a.data_ptr() % 16 or result.data_ptr() % 16 or T.data_ptr() % 4:
        raise B200DCTError("image buffers must be 16-byte aligned")
    with torch.cuda.device(a.device):
        torch.cuda.current_stream().synchronize()  # the wrappers run on the legacy default stream
        fn(a.data_ptr(), int(H), int(W), T.data_ptr(), result.data_ptr())


def dct_all_blocks_cuda(image_matrix, img_height, img_width, transform_matrix, result):
    """main_newAppr.cu:252 / main_fastAppr.cu:303.  Leaves image_matrix holding image-128."""
    _compat_call(compat_lib().b200dct_compat_dct, image_matrix, img_height, img_width, transform_matrix, result)


def idct_all_blocks_cuda(image_matrix, img_height, img_width, transform_matrix, result):
    """main_newAppr.cu:293 / main_fastAppr.cu:361."""
    _compat_call(compat_lib().b200dct_compat_idct, image_matrix, img_height, img_width, transform_matrix, result)


def dct_all_blocks(image_matrix, img_height, img_width, transform_matrix, result, handle=None):
    """main_cublass.cu:197 / main_cublass_2.cu:197; the cuBLAS handle is ignored."""
    _compat_call(compat_lib().b200dct_compat_dct, image_matrix, img_height, img_width, transform_matrix, result)


def idct_all_blocks(image_matrix, img_height, img_width, transform_matrix, result, handle=None, dequant_in_place=False):
    """main_cublass.cu:265 (const input) / main_cublass_2.cu:257 (input dequantised in place
    when dequant_in_place=True, the v2 behaviour)."""
    fn = compat_lib().b200dct_compat_idct_inplace_dequant if dequant_in_place else compat_lib().b200dct_compat_idct
    _compat_call(fn, image_matrix, img_height, img_width, transform_matrix, result)
