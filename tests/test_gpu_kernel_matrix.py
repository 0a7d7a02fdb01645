"""GPU: every compiled kernel, reached through the public API and checked against the oracle, with a launch
ledger that proves which kernel each cell ran.

The library picks one of 182 kernels at run time (tests/kernel_ledger.py reads the inventory from the built
libraries).  Each cell below is one call through the Python API: it names the kernel it must launch, runs the
call under torch.profiler, asserts that this kernel -- and no other kernel of the libraries -- ran, and
compares the output with a reference the suite already trusts:
  * exact arithmetic (Haweel's T with the chain inverse, dense T as ordered chains): the oracle, bit for bit;
    int16 and zig-zag coefficients are the oracle's coefficients clipped to [-32768, 32767];
  * the factored inverse (u8 output of Haweel's T) and the even/odd kernels of a symmetric dense T: the float64
    reference of tests/f64ref.py with its derived bound (these cells carry the `factored` marker; every plan
    sets its modes explicitly, so the result does not depend on the environment);
  * colour: oracle.roundtrip_rgb and tests/rgb420_ref.py; metrics: oracle.metrics; coded sizes:
    oracle.coded_bits.
Every output is pre-filled with a sentinel inside a larger buffer; the guard rows and columns around it
must survive the call, and inputs must be unchanged.

Layout: H = 40 (H/8 = 5 block rows: the last CTA row of the direct family, 4 block rows per CTA, has invalid
threads); W = 512 (W/8 = 64: full zig-zag warps and full 256-pixel TMA tiles) or 544 (a partial last warp and
tile).  An f32 plane is placed 32-byte aligned ('a'), at a 16-byte offset ('h') or with a pitch that is only a
multiple of 16 bytes ('p'); the direct family moves 32-byte aligned f32 planes with 256-bit accesses, one bit
per plane (DirectParams::v8), and the v8 cells set and clear each bit with the other two fixed.

Deep twins (DEEP): every cell of the TMA family again at W = 2080 (a partial last tile column) and an H derived from
the device's SM count and the cell's CTA size, so that every warp of the persistent kernel works through several
tiles: run tickets, then single tickets, a tail that starts on an odd remainder (tests/tma_depth.py).  A deep cell
reads its launch's grid and block from the profiler trace and asserts that regime, then checks the whole image.

The last tests assert that passing cells launched every kernel of the inventory, and passing deep cells every
kernel of the TMA family.
"""
from __future__ import annotations

import ctypes
import zlib
from typing import NamedTuple

import numpy as np
import pytest

import f64ref as R
import kernel_ledger as KL
import rgb420_ref
import tma_depth as D

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

F32 = np.float32
H0 = 40
FULL, PART = 512, 544
# 28 << 20 pixels, exactly TMA_BIG_PIXELS of b200dct.cu: the smallest image at which AUTO runs an f32 round trip of
# Haweel's T on the TMA family (prefers_tma compares with >=).  Far above the other cells, but no smaller size
# reaches AUTO's TMA choice.
BIG = (3584, 8192)
IRREGULAR = 0x8142_2418_1824_C3FF  # a runtime keep mask that is no zig-zag prefix
SENT = {torch.float32: 0x7FC0DEAD, torch.uint8: 0xA5, torch.int16: 0x5A5A}
PATH = {"direct": 1, "tma": 2, "auto": 0}

# kernels that no host path can select: none
ALLOWLIST: dict[str, str] = {}

LAUNCHED: dict[str, str] = {}   # key -> first passing cell that launched it
CELLS_PASSED: set[str] = set()
DEEP_LAUNCHED: dict[str, str] = {}   # the same for the deep cells
DEEP_PASSED: set[str] = set()


# ---------------------------------------------------------------- plans
class Unit(NamedTuple):
    T: str        # haweel | dct2 | rand (a non-symmetric dense T)
    Q: str        # jpeg | int (2 x jpeg) | div (0.37 x jpeg: no exact fast division)
    keep: str     # all | irr (IRREGULAR) | zz8 (first 8 zig-zag) | k6 .. k10 (compiled masks, round trips)
    dense: int    # DENSE_CHAIN (1) or DENSE_SYMMETRIC (2)
    tk: int       # TK_DENSE 0, TK_HAWEEL 1, TK_DENSE_SYM 2
    qm: int       # Q_IMM 0, Q_PARAM 1, Q_PARAM_DIV 2, Q_IMM_K6.. 3..7


UNITS = {
    "s0": Unit("haweel", "jpeg", "all", 1, 1, 0),
    "s1": Unit("haweel", "int", "all", 1, 1, 1),
    "s1m": Unit("haweel", "jpeg", "irr", 1, 1, 1),
    "s1z": Unit("haweel", "jpeg", "zz8", 1, 1, 1),    # not for round trips: k = 8 is a compiled mask there
    "s2": Unit("haweel", "div", "all", 1, 1, 2),
    "s2m": Unit("haweel", "div", "irr", 1, 1, 2),
    "d1": Unit("rand", "jpeg", "all", 1, 0, 1),
    "d1c": Unit("dct2", "int", "irr", 1, 0, 1),       # the DCT-II as ordered chains
    "d2": Unit("rand", "div", "all", 1, 0, 2),
    "d2c": Unit("dct2", "div", "all", 1, 0, 2),
    "y1": Unit("dct2", "jpeg", "all", 2, 2, 1),
    "y1m": Unit("dct2", "int", "irr", 2, 2, 1),
    "y2": Unit("dct2", "div", "all", 2, 2, 2),
    **{f"k{k}": Unit("haweel", "jpeg", f"k{k}", 1, 1, k - 3) for k in range(6, 11)},
}


def rand_T():
    return np.random.default_rng(8).uniform(-0.5, 0.5, 64).astype(F32)


def unit_arrays(oracle, u: Unit):
    T = {"haweel": oracle.haweel_T(), "dct2": oracle.dct2_T(), "rand": rand_T()}[u.T]
    Q = {"jpeg": oracle.jpeg_Q(), "int": (oracle.jpeg_Q() * F32(2)).astype(F32),
         "div": (oracle.jpeg_Q() * F32(0.37)).astype(F32)}[u.Q]
    if u.keep == "all":
        keep = oracle.ALL_COEFFS
    elif u.keep == "irr":
        keep = IRREGULAR
    else:
        keep = oracle.zigzag_mask(int(u.keep.lstrip("kz")))
    return T, Q, keep


def make_plan(dct, oracle, u: Unit, path: str, factored: bool):
    T, Q, keep = unit_arrays(oracle, u)
    plan = dct.Plan(T=None if u.T == "haweel" else T, Q=Q, keep=keep, path=PATH[path],
                    inverse=dct.api.INVERSE_FACTORED if factored else dct.api.INVERSE_EXACT, dense=u.dense)
    assert plan.kernel_kind == u.tk
    return plan, T, Q, keep


# ---------------------------------------------------------------- guarded buffers
class Buf:
    """A plane (H, W) -- or a zig-zag stream (H/8, W/8, 64) -- inside a larger buffer filled with a sentinel.
    align: 'a' 32-byte aligned, 'h' 16-byte offset, 'p' pitch a multiple of 16 but not of 32 bytes."""

    def __init__(self, H, W, dtype, align="a", data=None, zigzag=False):
        if zigzag:
            self.frame = torch.full((H // 8 + 2, W // 8 + 2, 64), SENT[torch.int16], dtype=torch.int16, device="cuda")
            self.view = self.frame[1:-1, 1:-1]
        else:
            es = torch.tensor([], dtype=dtype).element_size()
            g = 32 // es
            off = g // 2 if align == "h" else g
            extra = 16 // es if align == "p" else 0
            self.frame = torch.empty((H + 2, W + 2 * g + extra), dtype=dtype, device="cuda")
            self._bits(self.frame).fill_(SENT[dtype])
            self.view = self.frame[1:H + 1, off:off + W]
        if data is not None:
            self.view.copy_(torch.from_numpy(np.ascontiguousarray(data)).cuda())
        self.mask = torch.zeros(self.frame.shape, dtype=torch.bool, device="cuda")
        if zigzag:
            self.mask[1:-1, 1:-1] = True
        else:
            self.mask[1:H + 1, off:off + W] = True
        self.before = self.frame.clone()

    @staticmethod
    def _bits(t):
        return t.view(torch.int32) if t.dtype == torch.float32 else t

    def guards_intact(self) -> bool:
        a, b = self._bits(self.frame), self._bits(self.before)
        return torch.equal(a[~self.mask], b[~self.mask])

    def unchanged(self) -> bool:
        return torch.equal(self._bits(self.frame), self._bits(self.before))

    def host(self):
        torch.cuda.synchronize()
        return self.view.cpu().numpy()


def bits(a):
    return a.view(np.uint32) if a.dtype == np.float32 else a


def clip16(C):
    return np.clip(C, -32768, 32767)


def as_coef_plane(got, kind):
    """A coefficient buffer of the kernel as an f32 (H, W) plane."""
    return R.unzigzag(got) if kind == "zz" else got.astype(F32)


def want_coef(oracle, C, kind):
    """The expected contents of a coefficient buffer of kind f32 / i16 / zz for oracle coefficients C."""
    if kind == "f32":
        return C
    if kind == "i16":
        return clip16(C).astype(np.int16)
    return oracle.zigzag_i16(clip16(C).astype(F32))


def equal(got, want):
    return np.array_equal(bits(np.ascontiguousarray(got)), bits(np.ascontiguousarray(want)))


# ---------------------------------------------------------------- the launch ledger
@pytest.fixture(scope="session")
def inventory():
    if KL.tool("cuobjdump") is None or KL.tool("cu++filt") is None:
        pytest.skip("no cuobjdump / cu++filt in CUDA_HOME or on PATH: no kernel inventory")
    return KL.inventory()


def launched_by(inventory, fn, geometry=False):
    """Run fn() under torch.profiler (CUDA activity only); the set of inventory keys it launched, and with
    `geometry` the (name, grid, block) of every kernel from the exported trace (else None)."""
    from torch.profiler import ProfilerActivity, profile

    if geometry:
        res, prof, geo = D.profiled(fn)
    else:
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            D.warm_up()
            res = fn()
            torch.cuda.synchronize()
        geo = None
    keys = {KL.canonical(e.name) for e in prof.events()}
    return res, keys & set(inventory), geo


def expect_launch(inventory, cell_id, want, fn, deep_tiles=None):
    """deep_tiles: the tile count of a deep cell, whose k_tma launch must put every warp past two rounds (R3)."""
    want = {want} if isinstance(want, str) else set(want)
    assert want <= set(inventory), f"{cell_id}: expected kernels {want - set(inventory)} are not in the inventory"
    res, got, geo = launched_by(inventory, fn, geometry=deep_tiles is not None)
    assert got == want, f"{cell_id}: launched {sorted(got)}, expected {sorted(want)}"
    if deep_tiles is not None:
        key, grid, block = D.tma_launch(geo, KL.canonical)
        assert deep_tiles > 2 * grid * (block // 32) and D.regime(deep_tiles, grid, block) == "R3", \
            f"{cell_id}: {deep_tiles} tiles on grid {grid} x {block // 32} warps is not the deep regime"
    return res, want


def passed(cell_id, keys, deep=False):
    (DEEP_PASSED if deep else CELLS_PASSED).add(cell_id)
    for k in keys:
        (DEEP_LAUNCHED if deep else LAUNCHED).setdefault(k, cell_id)


# ---------------------------------------------------------------- the planar cells
class Cell(NamedTuple):
    entry: str       # fwd | inv | rt | met | batch
    family: str      # direct | tma | auto
    unit: str
    pix: str         # f32 | u8
    coef: str | None  # fwd: output kind; inv: input kind; rt / met: optional plane (f32 | i16 | zz)
    inv: str         # x: EXACT, f: FACTORED
    layout: str = "aaa"  # alignment of the (input, output, coefficient) f32 planes
    W: int = PART
    H: int = H0
    deep: bool = False   # H is the deep height of the device and the cell's CTA size (tma_depth.deep_height)

    @property
    def id(self):
        return (f"{self.entry}-{self.family}-{self.unit}-{self.pix}-{self.coef or 'none'}-{self.inv}-{self.layout}-"
                f"{'deep' if self.deep else self.H}x{self.W}")


MODE = {"fwd": 0, "inv": 1, "rt": 2, "met": 2, "batch": 2}


def finv_of(c: Cell) -> int:
    """The factored inverse: u8 output of Haweel's T, not with a compiled mask (those kernels keep the chains)."""
    u = UNITS[c.unit]
    return int(c.inv == "f" and c.entry != "fwd" and c.pix == "u8" and u.tk == 1 and u.qm <= 2)


def expected_kernel(c: Cell) -> str:
    u = UNITS[c.unit]
    pix = 0 if c.pix == "f32" else 1
    met = int(c.entry == "met")
    finv = finv_of(c)
    fam = "tma" if c.family in ("tma", "auto") else "direct"
    if fam == "tma":
        return f"k_tma<{MODE[c.entry]},{u.tk},{u.qm},{pix},{finv},{met}>"
    return f"k_direct<{MODE[c.entry]},{u.tk},{u.qm},{pix},{met},{finv}>"


def reassociated(c: Cell) -> bool:
    """Checked against the float64 bound: the even/odd kernels of a symmetric dense T and the factored inverse."""
    return UNITS[c.unit].tk == 2 or finv_of(c) == 1


def planar_cells():
    cells = []
    # Haweel's T: the quantiser units s0 (JPEG table as immediates), s1 (runtime table or mask), s2 (IEEE division)
    direct_rows = [("fwd", "f32", "f32", "x"), ("fwd", "u8", "zz", "x"), ("fwd", "f32", "i16", "x"),
                   ("inv", "f32", "i16", "x"), ("inv", "u8", "zz", "x"), ("inv", "u8", "f32", "f"), ("inv", "f32", "zz", "x"),
                   ("rt", "f32", "zz", "x"), ("rt", "u8", "i16", "x"), ("rt", "u8", None, "f"), ("rt", "f32", None, "x"),
                   ("met", "f32", "zz", "x"), ("met", "u8", "f32", "x"), ("met", "u8", "zz", "f")]
    tma_rows = [("fwd", "f32", "f32", "x"), ("fwd", "u8", "i16", "x"), ("inv", "f32", "i16", "x"), ("inv", "u8", "f32", "x"),
                ("inv", "u8", "i16", "f"), ("rt", "f32", "i16", "x"), ("rt", "u8", "f32", "x"), ("rt", "u8", None, "f"),
                ("met", "f32", None, "x"), ("met", "f32", "i16", "x")]
    for fam, rows in (("direct", direct_rows), ("tma", tma_rows)):
        for n, unit in enumerate(("s0", "s1", "s2")):
            for i, (e, pix, coef, inv) in enumerate(rows):
                cells.append(Cell(e, fam, unit, pix, coef, inv, W=FULL if (i + n) % 2 else PART))
        # runtime masks on s1 / s2, the factored inverse with them
        for unit in ("s1m", "s2m"):
            cells += [Cell("rt", fam, unit, "u8", None, "f"), Cell("inv", fam, unit, "u8", "f32", "f", W=FULL),
                      Cell("met", fam, unit, "f32", None, "x")]
        cells += [Cell("fwd", fam, "s1z", "u8", "f32" if fam == "tma" else "zz", "x"),
                  Cell("inv", fam, "s1z", "u8", "i16", "f", W=FULL)]
        if fam == "direct":
            cells += [Cell("met", fam, "s1z", "u8", "zz", "f", W=FULL), Cell("met", fam, "s1m", "u8", "i16", "f"),
                      Cell("met", fam, "s2m", "u8", "zz", "f", W=FULL)]
    # dense T: ordered chains (d1 / d2, a random T or the DCT-II) and the even/odd kernels (y1 / y2)
    dense_direct = [("fwd", "f32", "i16"), ("fwd", "u8", "zz"), ("inv", "f32", "zz"), ("inv", "u8", "f32"), ("inv", "u8", "i16"),
                    ("rt", "f32", "f32"), ("rt", "u8", None), ("rt", "u8", "zz"), ("met", "f32", None), ("met", "u8", "zz")]
    dense_tma = [("fwd", "f32", "i16"), ("fwd", "u8", "f32"), ("inv", "f32", "f32"), ("inv", "u8", "i16"),
                 ("rt", "f32", "i16"), ("rt", "u8", None), ("rt", "u8", "f32")]
    for fam, rows in (("direct", dense_direct), ("tma", dense_tma)):
        for n, unit in enumerate(("d1", "d2", "d1c", "d2c", "y1", "y2", "y1m")):
            for i, (e, pix, coef) in enumerate(rows):
                if unit in ("d1c", "d2c", "y1m") and i % 2:
                    continue                      # the second T / table of a unit: every other row
                cells.append(Cell(e, fam, unit, pix, coef, "x", W=FULL if (i + n) % 2 else PART))
    # compiled retained-coefficient masks (round trips of the JPEG table, first k zig-zag coefficients)
    for fam in ("direct", "tma"):
        for k in range(6, 11):
            cells.append(Cell("rt", fam, f"k{k}", "f32", "f32" if k % 2 else None, "x", W=FULL if k % 2 else PART))
            cells.append(Cell("rt", fam, f"k{k}", "u8", ("zz" if fam == "direct" else "i16") if k % 2 == 0 else None, "f",
                              W=PART if k % 2 else FULL))
    # 256-bit accesses: each v8 bit of the direct family set and cleared with the other two fixed
    for lay in ("aaa", "haa", "aha", "aah", "hhh", "pap", "app", "hha"):
        cells.append(Cell("rt", "direct", "s0", "f32", "f32", "x", layout=lay, W=FULL if lay[0] == "a" else PART))
    for lay in ("ha", "ah", "pa", "ap", "hh"):
        cells.append(Cell("fwd", "direct", "s2", "f32", "f32", "x", layout=lay + "a"))
        cells.append(Cell("inv", "direct", "d1", "f32", "f32", "x", layout=lay + "a", W=FULL))
    for lay in ("aah", "aha", "haa"):
        cells.append(Cell("met", "direct", "s1", "f32", "f32", "x", layout=lay))
    # zig-zag streams: full warps (cooperative) and a partial last warp (per lane), with and without metrics
    for W in (FULL, PART):
        cells += [Cell("rt", "direct", "s0", "u8", "zz", "x", W=W), Cell("met", "direct", "s0", "f32", "zz", "x", W=W),
                  Cell("met", "direct", "s0", "u8", "zz", "f", W=W), Cell("fwd", "direct", "s0", "f32", "zz", "x", W=W),
                  Cell("inv", "direct", "s0", "u8", "zz", "f", W=W)]
    # batches (the RT kernels with the image table) and AUTO at a size where it picks the TMA family
    cells += [Cell("batch", "direct", "s0", "f32", None, "x"), Cell("batch", "direct", "s2", "u8", None, "f", W=FULL),
              Cell("batch", "direct", "y1", "u8", None, "x"), Cell("rt", "auto", "s0", "f32", None, "x", H=BIG[0], W=BIG[1])]
    return list({c.id: c for c in cells}.values())     # a cell listed twice runs once


PLANAR = planar_cells()


def deep_cells():
    """A twin of every TMA-family cell at the deep width; its height is chosen on the device."""
    return list({d.id: d for d in (c._replace(W=D.DEEP_W, H=0, deep=True) for c in PLANAR if c.family == "tma")}.values())


DEEP = deep_cells()


def cta_warps(c: Cell) -> int:
    """Warps per CTA of the cell's k_tma launch (see tma_depth.cta_warps)."""
    coef = {"f32": "f32", "i16": "i16", None: None}[c.coef]
    planes = {"fwd": [c.pix, coef], "inv": [coef, c.pix]}.get(c.entry, [c.pix, c.pix] + ([coef] if coef else []))
    return D.cta_warps(c.pix, UNITS[c.unit].tk, planes, metrics=c.entry == "met")


def sm_count() -> int:
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _param(c: Cell):
    marks = [pytest.mark.factored] if reassociated(c) else []
    return pytest.param(c, id=c.id, marks=marks)


def image(oracle, c: Cell, seed):
    return oracle.rand_image(c.H, c.W, seed) if c.pix == "f32" else oracle.rand_image_u8(c.H, c.W, seed)


def kernel_coefs(dct, c, img_buf, plan):
    """The coefficients of the cell's plan on its image, from an unprofiled forward call of the same family
    (even/odd kernels: the forward of the round trip is the same code)."""
    coef = torch.empty(img_buf.view.shape, dtype=torch.float32, device="cuda")
    dct.forward(img_buf.view, coef, plan=plan)
    torch.cuda.synchronize()
    return coef.cpu().numpy()


def check_metrics(oracle, what, got, x, y):
    """(MSE, PEEN) of a call against oracle.metrics(x, y).  u8: the library's sums are exact integers, so MSE is
    the same double and PEEN the same expression of the same two integers; f32: within 1e-6 relative."""
    mse, peen = got
    wm, wp = oracle.metrics(x, y)
    if x.dtype == np.uint8:
        sse = float(((x.astype(np.int64) - y.astype(np.int64)) ** 2).sum())
        energy = float((x.astype(np.int64) ** 2).sum())
        assert mse == wm and mse == sse / x.size, f"{what}: MSE {mse!r} vs {wm!r}"
        assert peen == (100.0 * (sse / energy) ** 0.5 if energy > 0 else 0.0), f"{what}: PEEN {peen!r}"
        assert peen == pytest.approx(wp, rel=1e-15), f"{what}: PEEN {peen!r} vs {wp!r}"
    else:
        assert mse == pytest.approx(wm, rel=1e-6) and peen == pytest.approx(wp, rel=1e-6), f"{what}: {got} vs {(wm, wp)}"


def check_pixels(what, got, C, T, Q, exact_want=None):
    if exact_want is not None:
        assert equal(got, exact_want), f"{what}: pixels differ from the oracle"
        return
    ch = D.check_pixels_banded(got, C, T, Q)
    assert ch.bad == 0, f"{what}: pixels outside the float64 bound: {ch}"


@pytest.mark.parametrize("c", [_param(c) for c in PLANAR + DEEP])
def test_cell(dct, oracle, inventory, c: Cell):
    u = UNITS[c.unit]
    deep_tiles = None
    if c.deep:
        c = c._replace(H=D.deep_height(sm_count(), cta_warps(c), c.W))
        deep_tiles = D.ntiles(c.H, c.W)
    launch = lambda key, fn: expect_launch(inventory, c.id, key, fn, deep_tiles)  # noqa: E731
    nthr = oracle.max_threads()
    plan, T, Q, keep = make_plan(dct, oracle, u, c.family, c.inv == "f")
    Tn = None if u.T == "haweel" else T
    key = expected_kernel(c)
    exact = not reassociated(c)
    seed = zlib.crc32(c.id.encode()) % 1000 + 1
    img = image(oracle, c, seed)
    pdt = torch.float32 if c.pix == "f32" else torch.uint8
    lay = lambda i, dt: c.layout[i] if dt == torch.float32 else "a"   # noqa: E731
    cdt = {"f32": torch.float32, "i16": torch.int16, "zz": torch.int16, None: None}[c.coef]
    zz = c.coef == "zz"

    if c.entry == "batch":
        imgs = [image(oracle, c, seed + k) for k in range(3)]
        ins = [Buf(c.H, c.W, pdt, data=a) for a in imgs]
        outs = [Buf(c.H, c.W, pdt) for _ in imgs]
        _, keys = launch(key, lambda: dct.roundtrip_batch([b.view for b in ins], [o.view for o in outs], plan=plan))
        for a, i, o in zip(imgs, ins, outs):
            assert i.unchanged() and o.guards_intact()
            if exact:
                check_pixels(c.id, o.host(), None, T, Q, oracle.roundtrip(a, T=Tn, Q=Q, keep=keep))
            else:
                check_pixels(c.id, o.host(), kernel_coefs(dct, c, i, plan), T, Q)
        passed(c.id, keys, c.deep)
        return

    if c.entry == "fwd":
        src = Buf(c.H, c.W, pdt, lay(0, pdt), data=img)
        dst = Buf(c.H, c.W, cdt, lay(1, cdt), zigzag=zz)
        _, keys = launch(key, lambda: dct.forward(src.view, dst.view, plan=plan, zigzag=zz))
        assert src.unchanged() and dst.guards_intact(), f"{c.id}: input changed or guard overwritten"
        got = dst.host()
        if exact:
            assert equal(got, want_coef(oracle, oracle.dct(img.astype(F32), T=Tn, Q=Q, keep=keep, threads=nthr), c.coef)), c.id
        else:
            ch = D.check_quant_banded(as_coef_plane(got, c.coef), img, T, Q, keep)
            assert ch.bad == 0, f"{c.id}: {ch}"
        passed(c.id, keys, c.deep)
        return

    if c.entry == "inv":
        C = clip16(oracle.dct(img.astype(F32), T=Tn, Q=Q, keep=keep, threads=nthr))
        data = oracle.zigzag_i16(C) if zz else C.astype(np.int16) if c.coef == "i16" else C
        src = Buf(c.H, c.W, cdt, lay(0, cdt), data=data, zigzag=zz)
        dst = Buf(c.H, c.W, pdt, lay(1, pdt))
        _, keys = launch(key, lambda: dct.inverse(src.view, dst.view, plan=plan, zigzag=zz))
        assert src.unchanged() and dst.guards_intact(), f"{c.id}: input changed or guard overwritten"
        want = None
        if exact:
            P = oracle.idct(C, T=Tn, Q=Q, threads=nthr)
            want = P if c.pix == "f32" else oracle.to_u8(P)
        check_pixels(c.id, dst.host(), C, T, Q, want)
        passed(c.id, keys, c.deep)
        return

    # round trips, with or without fused metrics
    src = Buf(c.H, c.W, pdt, lay(0, pdt), data=img)
    out = Buf(c.H, c.W, pdt, lay(1, pdt))
    cb = Buf(c.H, c.W, cdt, lay(2, cdt), zigzag=zz) if c.coef else None
    cv = cb.view if cb else None
    if c.entry == "met":
        fn = lambda: dct.roundtrip_with_metrics(src.view, out.view, cv, plan=plan, zigzag=zz)  # noqa: E731
    else:
        fn = lambda: dct.roundtrip(src.view, out.view, cv, plan=plan, zigzag=zz)  # noqa: E731
    res, keys = launch(key, fn)
    assert src.unchanged() and out.guards_intact() and (cb is None or cb.guards_intact()), \
        f"{c.id}: input changed or guard overwritten"
    got = out.host()
    want_out = None
    if u.tk == 2:     # even/odd forward: the kernel's coefficients, within the bound of the exact ones
        C = as_coef_plane(cb.host(), c.coef) if cb is not None else kernel_coefs(dct, c, src, plan)
        ch = D.check_quant_banded(C, img, T, Q, keep)
        assert ch.bad == 0, f"{c.id}: coefficients {ch}"
    else:             # the forward is the chain: the oracle's coefficients
        want_out, C = oracle.roundtrip(img, T=Tn, Q=Q, keep=keep, want_coef=True, threads=nthr)
        if cb is not None:
            assert equal(cb.host(), want_coef(oracle, C, c.coef)), f"{c.id}: coefficients differ from the oracle"
    check_pixels(c.id, got, C, T, Q, want_out if exact else None)
    if c.entry == "met":
        mse, peen, nnz = res[1]
        check_metrics(oracle, c.id, (mse, peen), img, got)
        assert nnz == int(np.count_nonzero(C)), f"{c.id}: non-zero count {nnz} vs {int(np.count_nonzero(C))}"
    passed(c.id, keys, c.deep)


# ---------------------------------------------------------------- any size (k_any, k_any_u8)
ANY = [(u, pix, inv) for u in ("d1", "d2", "s0", "s1", "s2", "y1", "y2") for pix in ("f32", "u8") for inv in ("x",)] + \
      [(u, "u8", "f") for u in ("s0", "s1m", "s2")]


@pytest.mark.parametrize("unit,pix,inv", [pytest.param(*a, id="-".join(a), marks=[pytest.mark.factored] if a[0][0] == "y" or a[2] == "f"
                                                        else []) for a in ANY])
def test_any_cell(dct, oracle, inventory, unit, pix, inv):
    """roundtrip_any of a ragged image into a guarded view: one pass of the edge-replicating kernel."""
    u = UNITS[unit]
    plan, T, Q, keep = make_plan(dct, oracle, u, "auto", inv == "f")
    Tn = None if u.T == "haweel" else T
    H, W = 37, 101
    pdt = torch.float32 if pix == "f32" else torch.uint8
    rng = np.random.default_rng(len(unit) * 7 + len(pix))
    img = rng.integers(0, 256, (H, W)).astype(F32 if pix == "f32" else np.uint8)
    src, dst = Buf(H, W, pdt, data=img), Buf(H, W, pdt)
    finv = int(inv == "f")
    key = f"k_any<{u.tk},{u.qm},0,0>" if pix == "f32" else f"k_any_u8<{u.tk},{u.qm},{finv}>"
    cid = f"any-{unit}-{pix}-{inv}"
    _, keys = expect_launch(inventory, cid, key, lambda: dct.roundtrip_any(src.view, dst.view, plan=plan))
    assert dct.api.last_path() == "any"
    assert src.unchanged() and dst.guards_intact()
    padded = np.ascontiguousarray(np.pad(img, ((0, -H % 8), (0, -W % 8)), mode="edge"))
    got = dst.host()
    if u.tk != 2 and inv == "x":
        assert equal(got, oracle.roundtrip(padded, T=Tn, Q=Q, keep=keep)[:H, :W]), cid
    else:
        if u.tk == 2:
            C = kernel_coefs(dct, None, Buf(*padded.shape, pdt, data=padded), plan)
            Y, B = R.forward64(padded, T)
            assert R.check_quant(C, Y, B, Q, keep).bad == 0
        else:
            C = oracle.dct(padded.astype(F32), Q=Q, keep=keep)
        P, Bi = R.inverse64(C, T, Q)
        ch = R.check_u8(got, P[:H, :W], Bi[:H, :W]) if pix == "u8" else R.check_close(got, P[:H, :W], Bi[:H, :W])
        assert ch.bad == 0, f"{cid}: {ch}"
    passed(cid, keys)


# ---------------------------------------------------------------- colour (k_rgb*, k_rgb420*)
def rgb_plan(dct, oracle, qk, factored):
    """qk 0: every coefficient, fast division; 1: a runtime mask; 2: tables without an exact fast division."""
    Q, Qc, keep = oracle.jpeg_Q(), oracle.jpeg_Q_chroma(), oracle.ALL_COEFFS
    if qk == 1:
        keep = IRREGULAR
    if qk == 2:
        Q, Qc = (Q * F32(0.37)).astype(F32), (Qc * F32(0.37)).astype(F32)
    plan = dct.Plan(Q=Q, Qc=Qc, keep=keep, inverse=dct.api.INVERSE_FACTORED if factored else dct.api.INVERSE_EXACT)
    return plan, Q, Qc, keep


def rgb_image(H, W, seed):
    return np.random.default_rng(seed).integers(0, 256, (H, W, 3)).astype(np.uint8)


class RgbBuf:
    """An (H, W, 3) u8 image 8 pixels inside a sentinel frame (rows 8-byte aligned)."""

    def __init__(self, H, W, data=None):
        self.frame = torch.full((H + 2, W + 16, 3), 0xA5, dtype=torch.uint8, device="cuda")
        self.view = self.frame[1:H + 1, 8:W + 8]
        if data is not None:
            self.view.copy_(torch.from_numpy(data).cuda())
        self.before = self.frame.clone()
        self.mask = torch.zeros(self.frame.shape, dtype=torch.bool, device="cuda")
        self.mask[1:H + 1, 8:W + 8] = True

    def guards_intact(self):
        return torch.equal(self.frame[~self.mask], self.before[~self.mask])

    def unchanged(self):
        return torch.equal(self.frame, self.before)


def streams3(H, W, data=None):
    """(3, H/8, W/8, 64) int16 streams between two sentinel planes."""
    frame = torch.full((5, H // 8, W // 8, 64), 0x5A5A, dtype=torch.int16, device="cuda")
    if data is not None:
        frame[1:4] = torch.from_numpy(data).cuda()
    return frame, frame[1:4], frame.clone()


RGB = [("rt", qk, f, zz) for qk in range(3) for f in (0, 1) for zz in (0, 1)] + [("fwd", qk, 0, 1) for qk in range(3)] + \
      [("inv", 0, f, 1) for f in (0, 1)]


@pytest.mark.parametrize("entry,qk,f,zz", [pytest.param(*a, id=f"{a[0]}-q{a[1]}-f{a[2]}-zz{a[3]}",
                                                        marks=[pytest.mark.factored] if a[2] else []) for a in RGB])
def test_rgb_cell(dct, oracle, inventory, entry, qk, f, zz):
    import test_gpu_reassociated as RA

    H, W = H0, PART
    plan, Q, Qc, keep = rgb_plan(dct, oracle, qk, f)
    rgb = rgb_image(H, W, 10 * qk + f)
    want, coef3 = oracle.roundtrip_rgb(rgb, Q=Q, Qc=Qc, keep=keep, want_coef=True)
    want_zz = np.stack([oracle.zigzag_i16(clip16(coef3[c])) for c in range(3)])
    cid = f"rgb-{entry}-q{qk}-f{f}-zz{zz}"
    src = RgbBuf(H, W, rgb)
    out = RgbBuf(H, W)
    if entry == "rt":
        key = f"k_rgb<{qk},{f},{zz}>"
        frame, zs, before = streams3(H, W)
        _, keys = expect_launch(inventory, cid, key, lambda: dct.roundtrip_rgb(src.view, out.view, zs if zz else None, plan=plan))
    elif entry == "fwd":
        key = f"k_rgb_forward<{qk}>"
        frame, zs, before = streams3(H, W)
        _, keys = expect_launch(inventory, cid, key, lambda: dct.forward_rgb(src.view, zs, plan=plan))
    else:
        key = f"k_rgb_inverse<{f}>"
        frame, zs, before = streams3(H, W, want_zz)
        _, keys = expect_launch(inventory, cid, key, lambda: dct.inverse_rgb(zs, out.view, plan=plan))
    torch.cuda.synchronize()
    assert src.unchanged() and out.guards_intact()
    assert torch.equal(frame[0], before[0]) and torch.equal(frame[4], before[4]), f"{cid}: stream guard overwritten"
    if entry == "inv":
        assert torch.equal(frame, before), f"{cid}: input streams changed"
    if zz:
        assert np.array_equal(zs.cpu().numpy(), want_zz), f"{cid}: streams differ from the oracle"
    if entry != "fwd":
        got = out.view.cpu().numpy()
        if f:
            RA.check_rgb(oracle, cid, got, coef3, oracle.haweel_T(), (Q, Qc, Qc))
        else:
            assert np.array_equal(got, want), f"{cid}: RGB differs from the oracle"
    passed(cid, keys)


RGB420 = [("fwd", qk, 0) for qk in range(3)] + [("inv", 1, f) for f in (0, 1)]


@pytest.mark.parametrize("entry,qk,f", [pytest.param(*a, id=f"{a[0]}-q{a[1]}-f{a[2]}", marks=[pytest.mark.factored] if a[2] else [])
                                        for a in RGB420])
def test_rgb420_cell(dct, oracle, inventory, entry, qk, f):
    import test_gpu_rgb420 as T420

    H, W = 48, PART
    plan, Q, Qc, keep = rgb_plan(dct, oracle, qk, f)
    rgb = rgb_image(H, W, 20 + qk)
    want = rgb420_ref.forward_rgb420(oracle, rgb, Q, Qc, keep)
    cid = f"rgb420-{entry}-q{qk}-f{f}"
    shapes = ((H // 8, W // 8, 64), (H // 16, W // 16, 64), (H // 16, W // 16, 64))
    # the three streams back to back in one buffer, with a sentinel block before, between and after them
    sizes = [int(np.prod(s)) for s in shapes]
    buf = torch.full((sum(sizes) + 4 * 64,), 0x5A5A, dtype=torch.int16, device="cuda")
    views, o = [], 64
    for s, n in zip(shapes, sizes):
        views.append(buf[o:o + n].view(s))
        o += n + 64
    if entry == "inv":
        for v, w in zip(views, want):
            v.copy_(torch.from_numpy(w).cuda())
    before = buf.clone()
    src, out = RgbBuf(H, W, rgb), RgbBuf(H, W)
    if entry == "fwd":
        _, keys = expect_launch(inventory, cid, f"k_rgb420_forward<{qk}>", lambda: dct.forward_rgb420(src.view, tuple(views), plan=plan))
    else:
        _, keys = expect_launch(inventory, cid, f"k_rgb420_inverse<{f}>", lambda: dct.inverse_rgb420(tuple(views), out.view, plan=plan))
    torch.cuda.synchronize()
    assert src.unchanged() and out.guards_intact()
    mask = torch.ones_like(buf, dtype=torch.bool)
    o = 64
    for n in sizes:
        mask[o:o + n] = False
        o += n + 64
    assert torch.equal(buf[mask], before[mask]), f"{cid}: stream guard overwritten"
    if entry == "fwd":
        for c, (v, w) in enumerate(zip(views, want)):
            assert np.array_equal(v.cpu().numpy(), w), f"{cid}: stream {c} differs from the reference"
    else:
        assert torch.equal(buf, before), f"{cid}: input streams changed"
        got = out.view.cpu().numpy()
        if f:
            T420.check_factored(oracle, got, want, Q, Qc)
        else:
            assert np.array_equal(got, rgb420_ref.inverse_rgb420(oracle, want, Q, Qc)), f"{cid}: RGB differs from the reference"
    passed(cid, keys)


# ---------------------------------------------------------------- the tensor-core arm, metrics, coded size, self-test, compat
@pytest.mark.parametrize("fastdiv", [True, False])
def test_mma_cell(dct, oracle, inventory, fastdiv):
    T = oracle.dct2_T()
    Q = oracle.jpeg_Q() if fastdiv else (oracle.jpeg_Q() * F32(0.37)).astype(F32)
    plan = dct.Plan(T=T, Q=Q, dense=dct.api.DENSE_MMA)
    img = oracle.rand_image(H0, PART, 5)
    src, out, cb = Buf(H0, PART, torch.float32, data=img), Buf(H0, PART, torch.float32), Buf(H0, PART, torch.float32)
    cid = f"mma-{fastdiv}"
    _, keys = expect_launch(inventory, cid, f"k_mma<{int(fastdiv)}>", lambda: dct.roundtrip(src.view, out.view, cb.view, plan=plan))
    assert dct.api.last_path() == "mma"
    assert src.unchanged() and out.guards_intact() and cb.guards_intact()
    Y, B = R.forward64(img, T)
    C = cb.host()
    assert R.check_quant(C, Y, B, Q, dct.ALL_COEFFS, R.C_MMA).bad == 0
    P, Bi = R.inverse64(C, T, Q)
    assert R.check_close(out.host(), P, Bi, R.C_MMA).bad == 0
    passed(cid, keys)


@pytest.mark.parametrize("pix", ["f32", "u8"])
def test_metrics_cell(dct, oracle, inventory, pix):
    a = oracle.rand_image(H0, PART, 3) if pix == "f32" else oracle.rand_image_u8(H0, PART, 3)
    b = oracle.roundtrip(a)
    dt = torch.float32 if pix == "f32" else torch.uint8
    ra, rb = Buf(H0, PART, dt, data=a), Buf(H0, PART, dt, data=b)
    cid = f"metrics-{pix}"
    (mse, peen), keys = expect_launch(inventory, cid, "k_metrics<float>" if pix == "f32" else "k_metrics<unsigned char>",
                                      lambda: dct.metrics(ra.view, rb.view))
    assert ra.unchanged() and rb.unchanged()
    check_metrics(oracle, cid, (mse, peen), a, b)
    passed(cid, keys)


@pytest.mark.parametrize("table", [0, 1])
def test_coded_bits_cell(dct, oracle, inventory, table):
    zz = oracle.zigzag_i16(oracle.dct(oracle.rand_image(H0, PART, 9), Q=(oracle.jpeg_Q() * F32(0.5)).astype(F32)))
    b = Buf(H0, PART, torch.int16, data=zz, zigzag=True)
    cid = f"coded-{table}"
    got, keys = expect_launch(inventory, cid, "k_coded_bits", lambda: dct.coded_bits(b.view, table))
    assert b.unchanged()
    assert got == oracle.coded_bits(zz, table)
    passed(cid, keys)


def test_selftest_division_cell(dct, inventory):
    acc = torch.zeros(2, dtype=torch.int64, device="cuda")
    first = int(np.float32(1.0).view(np.uint32))
    rc, keys = expect_launch(inventory, "selftest", "k_selftest_div",
                             lambda: dct.lib().b200dct_selftest_division(16.0, first, 1 << 22, acc.data_ptr(), None))
    assert rc == 0 and acc.tolist() == [0, 0]
    passed("selftest", keys)


def test_compat_cell(dct, oracle, inventory):
    """cublasDCTv2's inverse: the fused inverse, then the element-wise in-place dequantisation of the compat library."""
    img = oracle.rand_image(48, 80, 3)
    C = oracle.dct(img)
    coef, rec, T = (torch.from_numpy(x).cuda() for x in (C, np.zeros_like(img), oracle.haweel_T()))
    # the compat library's state is per thread: pin its defaults (side effects on, transform fetched every call,
    # the JPEG table, every coefficient), with the timing printout off for this cell only
    L = dct.api.compat_lib()
    L.b200dct_compat_cache_transform(0)
    L.b200dct_compat_set_quant((ctypes.c_float * 64)(*oracle.jpeg_Q().tolist()))
    L.b200dct_compat_set_keep_mask(dct.ALL_COEFFS)
    L.b200dct_compat_set_options(1, 0)
    try:
        _, keys = expect_launch(inventory, "compat", {"k_direct<1,1,0,0,0,0>", "k_dequant_inplace"},
                                lambda: dct.idct_all_blocks(coef, 48, 80, T, rec, None, dequant_in_place=True))
    finally:
        L.b200dct_compat_set_options(1, 1)
    assert equal(rec.cpu().numpy(), oracle.idct(C))
    assert np.array_equal(coef.cpu().numpy(), C * np.tile(oracle.jpeg_Q().reshape(8, 8), (6, 10)))
    passed("compat", keys)


# ---------------------------------------------------------------- the ledger
N_CELLS = len(PLANAR) + len(ANY) + len(RGB) + len(RGB420) + 2 + 2 + 2 + 1 + 1


def test_zz_every_kernel_launched(request, inventory):
    """Every kernel of the inventory was launched by a passing cell, less ALLOWLIST."""
    if len(CELLS_PASSED) != N_CELLS:
        pytest.skip(f"{N_CELLS - len(CELLS_PASSED)} of {N_CELLS} cells did not run or did not pass: the ledger is incomplete")
    launched = set(LAUNCHED)
    print(f"launched {len(launched)} of {len(inventory)}")
    never = sorted(set(inventory) - launched)
    for k in never:
        print(f"  not launched: {k}  ({ALLOWLIST.get(k, 'NOT ALLOWLISTED')})")
    assert set(never) <= set(ALLOWLIST), f"kernels no passing cell launched: {sorted(set(never) - set(ALLOWLIST))}"
    assert not set(ALLOWLIST) & launched, f"allowlisted kernels that were launched: {sorted(set(ALLOWLIST) & launched)}"


def test_zz_every_tma_kernel_launched_at_depth(inventory):
    """Every k_tma kernel of the inventory was launched by a passing deep cell: each one's tile loop ran with
    several tiles per warp and was checked over the whole image."""
    if len(DEEP_PASSED) != len(DEEP):
        pytest.skip(f"{len(DEEP) - len(DEEP_PASSED)} of {len(DEEP)} deep cells did not run or did not pass: the ledger is incomplete")
    tma = sorted(k for k in inventory if k.startswith("k_tma<"))
    print(f"{len(tma)} TMA kernels, launched at depth by {len(DEEP_PASSED)} deep cells")
    for k in tma:
        print(f"  {k}  {DEEP_LAUNCHED.get(k, 'NOT LAUNCHED AT DEPTH')}")
    never = sorted(set(tma) - set(DEEP_LAUNCHED))
    assert not never, f"TMA kernels no passing deep cell launched: {never}"
