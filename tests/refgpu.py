"""Test helper: run the UNMODIFIED reference (oracle/_ref/libref_*.so, built by oracle/Makefile
where the reference's sources are present) on torch CUDA tensors, and the stored digests of the
CPU oracle's outputs (tests/golden/refgpu_digests.json) that stand in for it where it is not
built.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os
import re
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
DIGESTS = os.path.join(ROOT, "tests", "golden", "refgpu_digests.json")
VARIANTS = {"newappr": "libref_newappr.so", "fastappr": "libref_fastappr.so",
            "cublas": "libref_cublas.so", "cublas2": "libref_cublas2.so"}
_libs = {}


def available(variant: str = "newappr") -> bool:
    return os.path.exists(os.path.join(REF_DIR, VARIANTS[variant]))


def digest(a) -> str:
    """sha256 over dtype, shape and the raw bytes (C order) of a numpy array or torch tensor:
    equal digests mean equal bits, sign of zero included."""
    import numpy as np

    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def stored(case: str) -> dict:
    """Digests (and metrics) of the oracle's outputs for one case of make_ref_digests.py."""
    with open(DIGESTS) as f:
        return json.load(f)["cases"][case]


def load(variant: str) -> C.CDLL:
    if variant not in _libs:
        L = C.CDLL(os.path.join(REF_DIR, VARIANTS[variant]))
        L.ref_set_quant.argtypes = [C.POINTER(C.c_float)]
        for f in (L.ref_dct, L.ref_idct):
            f.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
            f.restype = None
        _libs[variant] = L
    return _libs[variant]


class capture_stdout:
    """Capture C-level stdout (the reference printf()s its own event timing)."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        self._tmp = tempfile.TemporaryFile(mode="w+b")
        os.dup2(self._tmp.fileno(), 1)
        self.text = ""
        return self

    def __exit__(self, *exc):
        import ctypes

        ctypes.CDLL(None).fflush(None)
        os.dup2(self._saved, 1)
        os.close(self._saved)
        self._tmp.seek(0)
        self.text = self._tmp.read().decode(errors="replace")
        self._tmp.close()
        return False


def _times(text: str, tag: str):
    return [float(x) for x in re.findall(tag + r" \(\d+,\d+\): ([0-9.]+) ms", text)]


def set_quant(variant: str, q) -> int:
    import numpy as np

    a = np.ascontiguousarray(q, np.float32).reshape(64)
    return load(variant).ref_set_quant((C.c_float * 64)(*a.tolist()))


def dct(variant: str, image, T, result=None):
    """result = reference dct_all_blocks*(image, H, W, T).  `image` (f32 CUDA tensor) is
    mutated to image-128, exactly as the reference does.  Returns (result, ms)."""
    import torch

    H, W = image.shape
    if result is None:
        result = torch.empty_like(image)
    torch.cuda.synchronize()
    with capture_stdout() as cap:
        load(variant).ref_dct(image.data_ptr(), H, W, T.data_ptr(), result.data_ptr())
        torch.cuda.synchronize()
    t = _times(cap.text, "DCT")
    return result, (t[-1] if t else float("nan"))


def idct(variant: str, coef, T, result=None):
    import torch

    H, W = coef.shape
    if result is None:
        result = torch.empty_like(coef)
    torch.cuda.synchronize()
    with capture_stdout() as cap:
        load(variant).ref_idct(coef.data_ptr(), H, W, T.data_ptr(), result.data_ptr())
        torch.cuda.synchronize()
    t = _times(cap.text, "IDCT")
    return result, (t[-1] if t else float("nan"))
