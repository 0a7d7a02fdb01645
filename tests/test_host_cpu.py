"""CPU suite: host logic, the C ABI surface, loud failure without a device.  No GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def m():
    import cuda_dct_idct_b200 as mod

    if not os.path.exists(mod.lib_path()):
        import __graft_entry__ as g

        g.build()
    return mod


def _declared(header):
    src = open(os.path.join(ROOT, "include", header)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b200dct_\w+)\s*\(", src)))


def test_c_abi_exports_every_declared_symbol(m):
    L = m.lib()
    names = _declared("b200dct.h")
    assert len(names) >= 18
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/b200dct.h but not exported"
    Lc = m.api.compat_lib()
    for n in [x for x in _declared("b200dct_compat.h") if x.startswith("b200dct_compat_")]:
        assert hasattr(Lc, n), n


def test_compat_exports_reference_mangled_names(m):
    # the reference's C++ entry points keep their mangled names (what main_*.o would reference)
    Lc = m.api.compat_lib()
    for sym in ("_Z19dct_all_blocks_cudaPfiiPKfS_", "_Z20idct_all_blocks_cudaPKfiiS0_Pf",
                "_Z14dct_all_blocksPfiiPKfS_P13cublasContext",
                "_Z15idct_all_blocksPKfiiS0_PfP13cublasContext",   # main_cublass.cu:37
                "_Z15idct_all_blocksPfiiPKfS_P13cublasContext"):   # main_cublass_2.cu:37
        assert hasattr(Lc, sym), sym


def test_reference_symbols_match_when_ref_built(m):
    ref = os.path.join(ROOT, "oracle", "_ref", "libref_newappr.so")
    if not os.path.exists(ref):
        pytest.skip("oracle/_ref not built")
    R = C.CDLL(ref)
    assert hasattr(R, "_Z19dct_all_blocks_cudaPfiiPKfS_") and hasattr(R, "_Z20idct_all_blocks_cudaPKfiiS0_Pf")


def test_plan_and_masks_without_gpu(m, oracle):
    p = m.Plan()
    assert p.is_sparse
    assert np.array_equal(p.quant(), oracle.jpeg_Q())
    p.set_transform(oracle.dct2_T())
    assert not p.is_sparse
    p.set_transform(oracle.haweel_T())
    assert p.is_sparse
    for k in range(0, 65):
        assert m.zigzag_mask(k) == oracle.zigzag_mask(k)
    with pytest.raises(m.B200DCTError):
        p.set_quant(np.zeros(64, np.float32))
    q = oracle.jpeg_Q() * 2
    p.set_quant(q)
    assert np.array_equal(p.quant(), q)


def test_argument_errors_and_no_cpu_fallback(m):
    import torch

    L = m.lib()
    p = m.Plan()
    buf = (C.c_float * 64)()
    addr = C.addressof(buf)
    assert addr % 16 == 0 or True
    # shape errors are detected before any device work
    assert L.b200dct_roundtrip(p._h, addr, 0, 32, addr, 0, 32, None, 0, 0, 8, 12, None) == -2
    assert L.b200dct_roundtrip(p._h, addr, 0, 16, addr, 0, 16, None, 0, 0, 8, 8, None) == -2  # pitch < row
    assert L.b200dct_roundtrip(p._h, None, 0, 32, addr, 0, 32, None, 0, 0, 8, 8, None) == -1
    assert L.b200dct_roundtrip(p._h, addr, 2, 32, addr, 0, 32, None, 0, 0, 8, 8, None) == -1   # i16 pixels
    assert L.b200dct_roundtrip(p._h, addr, 0, 32, addr, 1, 32, None, 0, 0, 8, 8, None) == -1   # mixed pixel dtypes
    # zig-zag coefficient stream: coefficient role only, pitch = bytes per block-row (>= (W/8)*128)
    big = (C.c_float * 256)()
    baddr = C.addressof(big) + (-C.addressof(big)) % 16
    assert L.b200dct_roundtrip(p._h, addr, 3, 128, addr, 0, 32, None, 0, 0, 8, 8, None) == -1  # stream as pixels
    assert L.b200dct_forward(p._h, baddr, 0, 64, baddr, 3, 128, None, 8, 16, None) == -2        # 2 blocks need 256 B
    assert L.b200dct_forward(p._h, baddr, 0, 64, baddr, 3, 264, None, 8, 16, None) == -3        # pitch not 16 B aligned
    assert L.b200dct_error_string(-4).decode().startswith("no usable CUDA device")
    ARG, SHAPE, ALIGN, NODEV = -1, -2, -3, -4
    a16 = baddr                       # 16-byte aligned, never dereferenced: every call below fails before device work
    dense = m.Plan(T=np.eye(8, dtype=np.float32))
    assert not dense.is_sparse
    # forward / inverse / roundtrip: NULL plan before shape, H and W positive multiples of 8, pitch >= row
    assert L.b200dct_roundtrip(None, a16, 0, 32, a16, 0, 32, None, 0, 0, 8, 12, None) == ARG
    for H, W in ((0, 8), (8, 0), (-8, 8), (12, 8)):
        assert L.b200dct_roundtrip(p._h, a16, 0, 32, a16, 0, 32, None, 0, 0, H, W, None) == SHAPE
    assert L.b200dct_forward(None, a16, 0, 32, a16, 0, 32, None, 8, 4, None) == ARG
    assert L.b200dct_forward(p._h, a16, 0, 32, a16, 0, 32, None, 4, 8, None) == SHAPE
    assert L.b200dct_inverse(None, a16, 0, 32, a16, 0, 32, 8, 12, None) == ARG
    assert L.b200dct_inverse(p._h, a16, 0, 32, a16, 0, 32, 8, 12, None) == SHAPE
    assert L.b200dct_inverse(p._h, a16, 0, 16, a16, 0, 32, 8, 8, None) == SHAPE                    # pitch < row
    # fused metrics: workspace and accumulator first, then the rules of roundtrip
    ws = L.b200dct_metrics_workspace_bytes(8, 8)
    assert L.b200dct_roundtrip_metrics(p._h, a16, 0, 32, a16, 0, 32, None, 0, 0, 8, 8, None, a16, ws, None) == ARG
    assert L.b200dct_roundtrip_metrics(p._h, a16, 0, 32, a16, 0, 32, None, 0, 0, 8, 8, a16, a16, ws - 1, None) == ARG
    assert L.b200dct_roundtrip_metrics(None, a16, 0, 32, a16, 0, 32, None, 0, 0, 8, 12, a16, a16, ws, None) == ARG
    assert L.b200dct_roundtrip_metrics(p._h, a16, 0, 32, a16, 0, 32, None, 0, 0, 8, 12, a16, a16, ws, None) == SHAPE
    # any size: non-positive sides are ARG, pitch < row SHAPE, element misalignment ALIGN
    assert L.b200dct_roundtrip_any(p._h, a16, 0, 28, a16, 28, 0, 7, None) == ARG
    assert L.b200dct_roundtrip_any(p._h, a16, 0, 24, a16, 28, 5, 7, None) == SHAPE
    assert L.b200dct_roundtrip_any(p._h, a16 + 2, 0, 28, a16, 28, 5, 7, None) == ALIGN
    assert L.b200dct_roundtrip_any(p._h, a16 + 2, 0, 24, a16, 28, 5, 7, None) == SHAPE           # pitch before alignment
    assert L.b200dct_roundtrip_any(p._h, a16, 2, 28, a16, 28, 5, 7, None) == ARG                 # i16 pixels
    # batch: arguments, then shape, then every image's planes; no images and valid arguments: nothing to do
    imgs = (C.c_void_p * 2)(a16, a16)
    assert L.b200dct_roundtrip_batch(None, 2, imgs, imgs, 0, 32, 32, 8, 12, None) == ARG
    assert L.b200dct_roundtrip_batch(p._h, 2, imgs, imgs, 2, 32, 32, 8, 12, None) == ARG          # i16 pixels
    assert L.b200dct_roundtrip_batch(p._h, 2, imgs, imgs, 0, 32, 32, 8, 12, None) == SHAPE
    assert L.b200dct_roundtrip_batch(p._h, 0, None, None, 0, 32, 32, 12, 8, None) == SHAPE
    assert L.b200dct_roundtrip_batch(p._h, 2, imgs, imgs, 0, 16, 32, 8, 8, None) == SHAPE          # pitch < row
    assert L.b200dct_roundtrip_batch(p._h, 2, imgs, imgs, 0, 40, 32, 8, 8, None) == ALIGN
    assert L.b200dct_roundtrip_batch(p._h, 0, None, None, 0, 32, 32, 8, 8, None) == 0
    # colour 4:4:4: NULL, shape, pitch, 8-byte RGB alignment, Haweel's T, stream alignment -- in this order
    zzb = 128
    for rc, args in ((ARG, (p._h, None, 24, a16, 24, None, 0, 8, 8)), (SHAPE, (p._h, a16, 24, a16, 24, None, 0, 8, 12)),
                     (SHAPE, (p._h, a16, 16, a16, 24, None, 0, 8, 8)), (ALIGN, (p._h, a16 + 4, 24, a16, 24, None, 0, 8, 8)),
                     (ALIGN, (p._h, a16, 28, a16, 24, None, 0, 8, 8)), (ARG, (dense._h, a16, 24, a16, 24, None, 0, 8, 8)),
                     (ALIGN, (p._h, a16, 24, a16, 24, a16 + 8, zzb, 8, 8)), (ALIGN, (p._h, a16, 24, a16, 24, a16, zzb - 16, 8, 8)),
                     (SHAPE, (dense._h, a16, 24, a16, 24, None, 0, 8, 12)), (ALIGN, (dense._h, a16 + 4, 24, a16, 24, None, 0, 8, 8)),
                     (ARG, (dense._h, a16, 24, a16, 24, a16 + 8, zzb, 8, 8))):
        assert L.b200dct_roundtrip_rgb(*args, None) == rc, (rc, args)
    assert L.b200dct_forward_rgb(p._h, a16, 24, None, zzb, 8, 8, None) == ARG
    assert L.b200dct_forward_rgb(p._h, a16, 24, a16, zzb, 12, 8, None) == SHAPE
    assert L.b200dct_forward_rgb(p._h, a16 + 4, 24, a16, zzb, 8, 8, None) == ALIGN
    assert L.b200dct_forward_rgb(dense._h, a16, 24, a16, zzb, 8, 8, None) == ARG
    assert L.b200dct_forward_rgb(p._h, a16, 24, a16 + 8, zzb, 8, 8, None) == ALIGN
    assert L.b200dct_forward_rgb(dense._h, a16, 24, a16 + 8, zzb, 8, 12, None) == SHAPE
    assert L.b200dct_inverse_rgb(p._h, None, zzb, a16, 24, 8, 8, None) == ARG
    assert L.b200dct_inverse_rgb(p._h, a16, zzb, a16, 16, 8, 8, None) == SHAPE
    assert L.b200dct_inverse_rgb(p._h, a16, zzb, a16, 28, 8, 8, None) == ALIGN
    assert L.b200dct_inverse_rgb(dense._h, a16, zzb, a16, 24, 8, 8, None) == ARG
    assert L.b200dct_inverse_rgb(p._h, a16, zzb + 8, a16, 24, 8, 8, None) == ALIGN
    # colour 4:2:0: sides multiples of 16, pitch, RGB and stream alignment, Haweel's T, then the grid (before the device)
    wide = (1 << 24) + 16                                                                         # 65537 CTAs across
    assert L.b200dct_forward_rgb420(p._h, a16, 48, a16, None, a16, 16, 16, None) == ARG
    assert L.b200dct_forward_rgb420(p._h, a16, 48, a16, a16, a16, 24, 16, None) == SHAPE
    assert L.b200dct_forward_rgb420(p._h, a16, 40, a16, a16, a16, 16, 16, None) == SHAPE
    assert L.b200dct_forward_rgb420(p._h, a16, 52, a16, a16, a16, 16, 16, None) == ALIGN
    assert L.b200dct_forward_rgb420(p._h, a16, 48, a16, a16 + 8, a16, 16, 16, None) == ALIGN
    assert L.b200dct_forward_rgb420(dense._h, a16, 48, a16, a16, a16, 16, 16, None) == ARG
    assert L.b200dct_forward_rgb420(p._h, a16, 3 * wide, a16, a16, a16, 16, wide, None) == SHAPE
    assert L.b200dct_forward_rgb420(dense._h, a16, 3 * wide, a16, a16, a16, 16, wide, None) == ARG
    assert L.b200dct_forward_rgb420(dense._h, a16, 48, a16, a16, a16 + 8, 16, 24, None) == SHAPE
    assert L.b200dct_inverse_rgb420(p._h, a16, a16, a16, None, 48, 16, 16, None) == ARG
    assert L.b200dct_inverse_rgb420(p._h, a16, a16, a16, a16, 48, 16, 8, None) == SHAPE
    assert L.b200dct_inverse_rgb420(p._h, a16, a16, a16 + 8, a16, 48, 16, 16, None) == ALIGN
    assert L.b200dct_inverse_rgb420(dense._h, a16, a16, a16, a16, 48, 16, 16, None) == ARG
    assert L.b200dct_inverse_rgb420(p._h, a16, a16, a16, a16, 3 * wide, 16, wide, None) == SHAPE
    # coded size: arguments, shape and pitch, alignment
    assert L.b200dct_zigzag_coded_bits(a16, 128, 8, 8, 2, a16, None) == ARG
    assert L.b200dct_zigzag_coded_bits(None, 128, 8, 12, 0, a16, None) == ARG
    assert L.b200dct_zigzag_coded_bits(a16, 128, 8, 12, 0, a16, None) == SHAPE
    assert L.b200dct_zigzag_coded_bits(a16, 128, 0, 8, 0, a16, None) == SHAPE
    assert L.b200dct_zigzag_coded_bits(a16, 112, 8, 8, 0, a16, None) == SHAPE
    assert L.b200dct_zigzag_coded_bits(a16, 136, 8, 8, 0, a16, None) == ALIGN
    assert L.b200dct_zigzag_coded_bits(a16 + 8, 128, 8, 12, 0, a16, None) == SHAPE
    # host pipeline: arguments, shape, pixel dtypes
    assert L.b200dct_roundtrip_host(None, a16, 0, a16, 0, 8, 12) == ARG
    assert L.b200dct_roundtrip_host(p._h, a16, 0, a16, 0, 8, 12) == SHAPE
    assert L.b200dct_roundtrip_host(p._h, a16, 0, a16, 0, -8, 8) == SHAPE
    assert L.b200dct_roundtrip_host(p._h, a16, 0, a16, 1, 8, 8) == ARG
    assert L.b200dct_roundtrip_host(p._h, a16, 0, a16, 1, 8, 12) == SHAPE
    assert L.b200dct_host_pipeline_submit(None, p._h, a16, 0, a16, 0, 8, 12, None) == ARG
    if not torch.cuda.is_available():
        # valid calls reach the device check on every entry point
        assert L.b200dct_forward(p._h, a16, 0, 32, a16, 0, 32, None, 8, 8, None) == NODEV
        assert L.b200dct_inverse(p._h, a16, 0, 32, a16, 0, 32, 8, 8, None) == NODEV
        assert L.b200dct_roundtrip(p._h, a16, 0, 32, a16, 0, 32, None, 0, 0, 8, 8, None) == NODEV
        assert L.b200dct_roundtrip_metrics(p._h, a16, 0, 32, a16, 0, 32, None, 0, 0, 8, 8, a16, a16, ws, None) == NODEV
        assert L.b200dct_roundtrip_any(p._h, a16, 0, 28, a16, 28, 5, 7, None) == NODEV
        assert L.b200dct_roundtrip_any(p._h, a16, 0, 32, a16, 32, 8, 8, None) == NODEV
        assert L.b200dct_roundtrip_batch(p._h, 2, imgs, imgs, 0, 32, 32, 8, 8, None) == NODEV
        assert L.b200dct_roundtrip_rgb(p._h, a16, 24, a16, 24, None, 0, 8, 8, None) == NODEV
        assert L.b200dct_roundtrip_rgb(p._h, a16, 24, a16, 24, a16, zzb, 8, 8, None) == NODEV
        assert L.b200dct_forward_rgb(p._h, a16, 24, a16, zzb, 8, 8, None) == NODEV
        assert L.b200dct_inverse_rgb(p._h, a16, zzb, a16, 24, 8, 8, None) == NODEV
        assert L.b200dct_forward_rgb420(p._h, a16, 48, a16, a16, a16, 16, 16, None) == NODEV
        assert L.b200dct_inverse_rgb420(p._h, a16, a16, a16, a16, 48, 16, 16, None) == NODEV
        assert L.b200dct_zigzag_coded_bits(a16, 128, 8, 8, 0, a16, None) == NODEV
        assert L.b200dct_roundtrip_host(p._h, a16, 0, a16, 0, 8, 8) == NODEV
        # the grid rule comes after the device check everywhere but 4:2:0
        assert L.b200dct_roundtrip(p._h, a16, 0, 4 * wide, a16, 0, 4 * wide, None, 0, 0, 8, wide, None) == NODEV
        assert L.b200dct_roundtrip_rgb(p._h, a16, 3 * wide, a16, 3 * wide, None, 0, 8, wide, None) == NODEV

        # valid arguments, no device: the product path refuses -- it never computes on the CPU
        a = np.zeros((8, 8), np.float32)
        b = np.zeros((8, 8), np.float32)
        rc = L.b200dct_roundtrip(p._h, a.ctypes.data - a.ctypes.data % 16 + 16 if a.ctypes.data % 16 else a.ctypes.data,
                                 0, 32, b.ctypes.data - b.ctypes.data % 16 + 16 if b.ctypes.data % 16 else b.ctypes.data,
                                 0, 32, None, 0, 0, 8, 8, None)
        assert rc in (-4, -3) or rc > 0
        assert rc != 0
        with pytest.raises(m.B200DCTError):
            m.roundtrip(torch.zeros(8, 8))          # CPU tensor: rejected
        with pytest.raises(m.B200DCTError):
            m.roundtrip_host(np.zeros((8, 8), np.float32))  # no device -> error, not a CPU result


def test_missing_library_fails_loudly(m, monkeypatch):
    monkeypatch.setattr(m.api, "_lib", None)
    monkeypatch.setattr(m.api, "lib_path", lambda name="libb200dct.so": "/nonexistent/" + name)
    with pytest.raises(m.B200DCTError, match="no CPU or PyTorch fallback"):
        m.api.lib()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "cuda-dct-idct_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")) or f == "Makefile":
                src = open(os.path.join(dp, f), errors="replace").read()
                assert "oracle" not in src.lower() or f in (), f"{f} mentions the oracle"
    for f in os.listdir(os.path.join(ROOT, "include")):
        assert "liboracle" not in open(os.path.join(ROOT, "include", f)).read()


def test_batch_images(m):
    for n in (0, 1, 7, 64, 65):
        for ws in (1, 2, 3, 8):
            shares = [m.batch_images(n, ws, r) for r in range(ws)]
            assert sorted(i for s in shares for i in s) == list(range(n))        # every image exactly once
            assert max(map(len, shares)) - min(map(len, shares)) <= 1
            assert all(i % ws == r for r, s in enumerate(shares) for i in s)     # image b on rank b mod world
    with pytest.raises(ValueError):
        m.batch_images(4, 2, 2)


def test_stripe_rows(m):
    for H in (8, 64, 8192, 32768, 72):
        for ws in (1, 2, 3, 4, 8, 16):
            spans = [m.stripe_rows(H, ws, r) for r in range(ws)]
            assert spans[0][0] == 0 and spans[-1][1] == H
            for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
                assert a1 == b0
            sizes = [b - a for a, b in spans]
            assert all(s % 8 == 0 for s in sizes) and max(sizes) - min(sizes) <= 8
    with pytest.raises(ValueError):
        m.stripe_rows(12, 2, 0)
    with pytest.raises(ValueError):
        m.stripe_rows(16, 2, 2)


def test_image_files_roundtrip_on_host(m, tmp_path):
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (37, 53)).astype(np.uint8)
    p = str(tmp_path / "a.pgm")
    m.imageio.save_gray(p, img)
    assert np.array_equal(m.imageio.load_gray(p), img)
    with open(p, "rb") as f:
        raw = f.read()
    with open(p, "wb") as f:                      # header with a comment line
        f.write(b"P5\n# made by a test\n53 37\n255\n" + raw[raw.index(b"255\n") + 4:])
    assert np.array_equal(m.imageio.load_gray(p), img)
    png = str(tmp_path / "a.png")
    m.imageio.save_gray(png, img)
    assert np.array_equal(m.imageio.load_gray(png), img)
    assert m.imageio.crop_to_blocks(img).shape == (32, 48)


def test_header_is_plain_c_and_links_from_c(m, tmp_path):
    """include/b200dct.h compiles as C99 (-pedantic -Werror) and a C program links against
    libb200dct.so: the boundary carries no C++ or torch types.  On a box without a GPU the
    program also checks that the host-buffer entry point refuses to run."""
    import shutil
    import subprocess

    import torch

    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    libdir = os.path.dirname(m.lib_path())
    exe = str(tmp_path / "abi_c99")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "abi_c99.c"), "-o", exe, "-L", libdir, "-lb200dct",
                           "-Wl,-rpath," + libdir])
    args = [exe] + (["--device"] if torch.cuda.is_available() else [])
    out = subprocess.run(args, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    assert "abi_c99 ok" in out.stdout


def test_module_cli_prints_usage():
    """`python -m cuda_dct_idct_b200` must reach the package's __main__ (ADVICE r1: it used to be a
    silent no-op because runpy resolves the name to the import shim)."""
    import subprocess
    import sys

    r = subprocess.run([sys.executable, "-m", "cuda_dct_idct_b200"], capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert r.returncode == 1 and "Usage:" in r.stderr
