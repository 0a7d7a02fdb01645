"""GPU: the persistent TMA kernels' tile loop in each CTA flavour, in each scheduler regime, captured, and in one
mixed programme; whole images against the oracle.

The five CTA flavours of k_tma (warps per CTA; csrc/dct_kernels.cuh tma_cta_threads, b200dct.cu run_tma):
  f32 Haweel 8, dense T 12, u8 with an f32 coefficient plane 14 (shared memory), u8 16, fused metrics 9.
Regimes (tests/tma_depth.py): R2 -- more tiles than warps, single tickets only; R3 -- run tickets, then single
tickets, every warp several tiles.  Each launch's grid and block are read back from the profiler trace and the
regime is asserted from them.

Captured launches own a ticket-counter pair for good; once a process has used up the capture pool, a captured
launch forced onto the TMA family takes the static split (tile += grid x warps).  Both run in a child process
(this file run as a script): the pool cannot be refilled.

Profiler sessions opened after a process has profiled and then captured a CUDA graph record no kernels (torch
2.11 with CUPTI).  The regime tests therefore run in a process that has not captured after profiling: no test
of this file captures in-process, and the file sorts right after tests/test_gpu_kernel_matrix.py, ahead of the
files that capture graphs in the test process.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys
from typing import NamedTuple

import numpy as np
import pytest

import kernel_ledger as KL
import tma_depth as D

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
PATH_TMA, INVERSE_EXACT, DENSE_CHAIN, DENSE_SYMMETRIC = 2, 1, 1, 2


class Flavour(NamedTuple):
    warps: int
    pix: str        # f32 | u8
    dense: bool     # a dense (random, non-symmetric) T as ordered chains, else Haweel's T
    coef: bool      # an f32 coefficient plane
    metrics: bool   # fused metrics


FLAVOURS = {
    "f32": Flavour(8, "f32", False, False, False),
    "dense": Flavour(12, "f32", True, False, False),
    "u8coef": Flavour(14, "u8", False, True, False),
    "u8": Flavour(16, "u8", False, False, False),
    "metrics": Flavour(9, "f32", False, False, True),
}
PLAIN = [n for n, f in FLAVOURS.items() if not f.metrics]


def rand_T():
    return np.random.default_rng(8).uniform(-0.5, 0.5, 64).astype(F32)


def sm_count() -> int:
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def height(f: Flavour, regime: str) -> int:
    return (D.deep_height if regime == "R3" else D.r2_height)(sm_count(), f.warps, D.DEEP_W)


def plan_of(dct, f: Flavour):
    return dct.Plan(T=rand_T() if f.dense else None, path=PATH_TMA, inverse=INVERSE_EXACT, dense=DENSE_CHAIN)


def image(oracle, pix, H, W, seed):
    return oracle.rand_image(H, W, seed) if pix == "f32" else oracle.rand_image_u8(H, W, seed)


def same(got, want) -> bool:
    return got.dtype == want.dtype and got.shape == want.shape and got.tobytes() == want.tobytes()


class Job:
    """One round trip of a flavour on device buffers; outputs pre-filled with a sentinel."""

    def __init__(self, dct, oracle, f: Flavour, H, W, seed):
        self.dct, self.f, self.plan = dct, f, plan_of(dct, f)
        self.img = image(oracle, f.pix, H, W, seed)
        self.x = torch.from_numpy(self.img).cuda()
        self.out = torch.empty_like(self.x)
        self.coef = torch.empty(self.x.shape, dtype=torch.float32, device="cuda") if f.coef else None
        self.clear()

    def clear(self):
        self.out.fill_(float("nan") if self.f.pix == "f32" else 0xA5)
        if self.coef is not None:
            self.coef.fill_(float("nan"))

    def __call__(self, stream=None):
        if self.f.metrics:
            return self.dct.roundtrip_with_metrics(self.x, self.out, plan=self.plan, stream=stream)[1]
        return self.dct.roundtrip(self.x, self.out, self.coef, plan=self.plan, stream=stream)

    def check(self, oracle, what, metrics=None):
        """The outputs against the oracle over the whole image."""
        torch.cuda.synchronize()
        out, coef = self.out.cpu().numpy(), None if self.coef is None else self.coef.cpu().numpy()
        want, C = oracle.roundtrip(self.img, T=rand_T() if self.f.dense else None, want_coef=True, threads=oracle.max_threads())
        assert same(out, want), f"{what}: pixels differ from the oracle at {np.argwhere(out != want)[:4].tolist()}"
        if coef is not None:
            assert same(coef, C), f"{what}: coefficients differ from the oracle"
        if metrics is not None:
            mse, peen, nnz = metrics
            wm, wp = oracle.metrics(self.img, out)
            assert mse == pytest.approx(wm, rel=1e-6) and peen == pytest.approx(wp, rel=1e-6), f"{what}: {metrics} vs {(wm, wp)}"
            assert nnz == int(np.count_nonzero(C)), f"{what}: non-zero count {nnz}"


def tma_regime(fn, H, W):
    """Run fn() under the profiler: (its result, the k_tma key, the regime of its launch, its warps per CTA)."""
    res, _, geo = D.profiled(fn)
    key, grid, block = D.tma_launch(geo, KL.canonical)
    return res, key, D.regime(D.ntiles(H, W), grid, block), block // 32


# ---------------------------------------------------------------- the scheduler regimes, once per CTA flavour
@pytest.mark.parametrize("regime", ["R2", "R3"])
@pytest.mark.parametrize("name", list(FLAVOURS))
def test_scheduler_regime(dct, oracle, name, regime):
    f = FLAVOURS[name]
    H, W = height(f, regime), D.DEEP_W
    job = Job(dct, oracle, f, H, W, seed=len(name) * 10 + len(regime))
    before = job.x.clone()
    res, key, got, warps = tma_regime(job, H, W)
    assert dct.api.last_path() == "tma"
    assert warps == f.warps, f"{name}: {warps} warps per CTA, expected {f.warps}"
    assert got == regime, f"{name} {key}: {D.ntiles(H, W)} tiles gave {got}, expected {regime}"
    assert torch.equal(job.x, before), f"{name}: input changed"
    job.check(oracle, f"{name}-{regime} {key}", metrics=res if f.metrics else None)


# ---------------------------------------------------------------- captured deep launches
def mismatches(oracle, job) -> int:
    """Pixels (and coefficients) of a job that differ from the oracle's, over the whole image."""
    torch.cuda.synchronize()
    out = job.out.cpu().numpy()
    want, C = oracle.roundtrip(job.img, T=rand_T() if job.f.dense else None, want_coef=True, threads=oracle.max_threads())
    n = int(np.count_nonzero(out.view(np.uint8) != want.view(np.uint8)))
    if job.coef is not None:
        n += int(np.count_nonzero(job.coef.cpu().numpy().view(np.uint32) != C.view(np.uint32)))
    return n


def child_captures():
    """Graph capture in a process of its own.  First, per flavour, one deep PATH_TMA round trip captured on a
    ticket-counter pair of its own, replayed twice with an ordinary deep launch in between.  Then the capture pool
    is used up, and deep PATH_TMA round trips captured after that take the static split; each is replayed twice.
    Every replay's output is compared with the oracle here; the result is a JSON line."""
    sys.path.insert(0, ROOT)
    import cuda_dct_idct_b200 as dct
    from oracle import oracle

    lib = dct.lib()
    s = torch.cuda.Stream()
    tiny = torch.zeros((8, 256), dtype=torch.float32, device="cuda")
    tiny_out = torch.empty_like(tiny)
    tiny_plan = dct.Plan(path=PATH_TMA)
    dct.roundtrip(tiny, tiny_out, plan=tiny_plan)     # the first ordinary call creates the pools
    torch.cuda.synchronize()
    res = {"own": {}, "static": {}}

    def capture(job):
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            job(s)
            path = dct.api.last_path()
        return g, path

    for name in PLAIN:
        f = FLAVOURS[name]
        H = height(f, "R3")
        cap, plain = Job(dct, oracle, f, H, D.DEEP_W, seed=31), Job(dct, oracle, f, H, D.DEEP_W, seed=32)
        g, path = capture(cap)
        r = {"path": path, "replays": []}
        for replay in (1, 2):
            cap.clear()
            g.replay()
            if replay == 1:
                plain()                               # stream-ordered after the replay, on an ordinary pair
                r["ordinary"] = mismatches(oracle, plain)
                r["ordinary_path"] = dct.api.last_path()
            r["replays"].append(mismatches(oracle, cap))
        res["own"][name] = r

    filler = torch.cuda.CUDAGraph()
    with torch.cuda.graph(filler, stream=s):
        for _ in range(int(lib.b200dct_capture_slots_left())):
            dct.roundtrip(tiny, tiny_out, plan=tiny_plan, stream=s)   # each captured TMA call takes a pair
    res["slots_left_after_fill"] = int(lib.b200dct_capture_slots_left())
    for name in ("f32", "u8", "dense"):
        f = FLAVOURS[name]
        job = Job(dct, oracle, f, height(f, "R3"), D.DEEP_W, seed=41)
        g, path = capture(job)
        r = {"path": path, "launches": dct.api.last_launch_count(), "replays": []}
        for replay in (1, 2):
            job.clear()
            g.replay()
            r["replays"].append(mismatches(oracle, job))
        res["static"][name] = r
    res["slots_left"] = int(lib.b200dct_capture_slots_left())
    return res


def test_captured_deep_launches(dct):
    """Run child_captures (this file as a script): a process that captures is not profiled afterwards by the other
    tests, and the capture pool it uses up is gone for good."""
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    # on a counter pair of its own: every replay exact, and so is the ordinary launch between them
    assert sorted(res["own"]) == sorted(PLAIN), res
    for name, o in res["own"].items():
        assert o["path"] == "tma" and o["ordinary_path"] == "tma", (name, o)
        assert o["replays"] == [0, 0] and o["ordinary"] == 0, (name, o)
    # the static split, with several tiles per warp
    assert res["slots_left_after_fill"] == 0 and res["slots_left"] == 0, res
    assert sorted(res["static"]) == ["dense", "f32", "u8"], res
    for name, o in res["static"].items():
        assert o == {"path": "tma", "launches": 1, "replays": [0, 0]}, (name, o)


# ---------------------------------------------------------------- one mixed-flavour programme
def test_mixed_flavour_programme(dct, oracle):
    """Round trips of every flavour on one stream without a synchronisation in between, dependent and
    independent, at a shape where each is deep; every output against the oracle applied in the same order.
    f32, dense and metrics CTAs take more than half an SM's shared memory (candidates for early tile loads
    across the launch boundary), u8 CTAs do not."""
    import f64ref as R

    nthr = oracle.max_threads()
    H, W = D.deep_height(sm_count(), 16, D.DEEP_W), D.DEEP_W     # deep for the largest CTA: deep for all
    api = dct.api
    haweel = dct.Plan(path=PATH_TMA, inverse=INVERSE_EXACT)
    T_sym = oracle.dct2_T()
    sym = dct.Plan(T=T_sym, path=PATH_TMA, inverse=INVERSE_EXACT, dense=DENSE_SYMMETRIC)
    assert sym.kernel_kind == 2
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    nan = lambda dt=torch.float32: torch.full((H, W), float("nan") if dt == torch.float32 else 0xA5, dtype=dt, device="cuda")  # noqa: E731

    a = oracle.rand_image(H, W, 51)
    u = oracle.rand_image_u8(H, W, 52)
    p = oracle.rand_image(H, W, 53)
    d, e = oracle.rand_image(H, W, 54), oracle.rand_image(H, W, 55)
    A, U, Pin, Dd, Ee = dev(a), dev(u), dev(p), dev(d), dev(e)
    B, Cs, Ccoef, Uo, P16, Pout, M, Do, Eo = nan(), nan(), nan(), nan(torch.uint8), nan(torch.int16), nan(), nan(), nan(), nan()
    P16.fill_(0x5A5A)
    acc = torch.zeros(3, dtype=torch.float64, device="cuda")
    nbytes = int(dct.lib().b200dct_metrics_workspace_bytes(H, W))
    ws = torch.empty(max(1, nbytes // 8), dtype=torch.float64, device="cuda")
    paths = []
    torch.cuda.synchronize()

    dct.roundtrip(A, B, plan=haweel)                                   # 1. f32 Haweel A -> B
    paths.append(api.last_path())
    dct.roundtrip(B, Cs, Ccoef, plan=sym)                              # 2. symmetric dense, reads B
    paths.append(api.last_path())
    dct.roundtrip(U, Uo, plan=haweel)                                  # 3. u8, unrelated
    paths.append(api.last_path())
    dct.forward(Pin, P16, plan=haweel)                                 # 4. forward to i16, inverse from it
    paths.append(api.last_path())
    dct.inverse(P16, Pout, plan=haweel)
    paths.append(api.last_path())
    bp, bdt, bpitch = api._plane(B)[:3]                                # 5. metrics, reads B (C ABI: no read-back)
    mp, mdt, mpitch = api._plane(M)[:3]
    rc = dct.lib().b200dct_roundtrip_metrics(haweel._h, bp, bdt, bpitch, mp, mdt, mpitch, None, api.F32, 0, H, W,
                                             acc.data_ptr(), ws.data_ptr(), nbytes, api._stream(None))
    assert rc == 0
    paths.append(api.last_path())
    dct.roundtrip(Dd, Do, plan=haweel)                                 # 6. two independent f32 round trips
    paths.append(api.last_path())
    dct.roundtrip(Ee, Eo, plan=haweel)
    paths.append(api.last_path())
    torch.cuda.synchronize()
    assert paths == ["tma"] * 8, paths

    host = lambda t: t.cpu().numpy()   # noqa: E731
    b, c1 = oracle.roundtrip(a, want_coef=True, threads=nthr)
    assert same(host(B), b), "1: f32 round trip"
    Cg = host(Ccoef)
    ch = D.check_quant_banded(Cg, b, T_sym, oracle.jpeg_Q(), R.ALL_COEFFS)
    assert ch.bad == 0, f"2: symmetric dense coefficients {ch}"
    ch = D.check_pixels_banded(host(Cs), Cg, T_sym, oracle.jpeg_Q())
    assert ch.bad == 0, f"2: symmetric dense pixels {ch}"
    assert same(host(Uo), oracle.roundtrip(u, threads=nthr)), "3: u8 round trip"
    Cp = np.clip(oracle.dct(p, threads=nthr), -32768, 32767)
    assert same(host(P16), Cp.astype(np.int16)), "4: forward to i16"
    assert same(host(Pout), oracle.idct(Cp, threads=nthr)), "4: inverse from i16"
    m, cm = oracle.roundtrip(b, want_coef=True, threads=nthr)
    assert same(host(M), m), "5: metrics round trip"
    sse, energy, nnz = acc.tolist()
    wm, wp = oracle.metrics(b, m)
    assert sse / (H * W) == pytest.approx(wm, rel=1e-6) and 100.0 * (sse / energy) ** 0.5 == pytest.approx(wp, rel=1e-6)
    assert int(nnz) == int(np.count_nonzero(cm)), "5: non-zero count"
    assert same(host(Do), oracle.roundtrip(d, threads=nthr)), "6: first independent round trip"
    assert same(host(Eo), oracle.roundtrip(e, threads=nthr)), "6: second independent round trip"
    for t, x in ((A, a), (U, u), (Pin, p), (Dd, d), (Ee, e)):
        assert same(host(t), x), "an input changed"


if __name__ == "__main__":
    print(json.dumps(child_captures()))
