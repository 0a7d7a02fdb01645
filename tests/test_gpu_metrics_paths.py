"""Launches that find no scheduler slot free: under stream capture once the capture pool is used up.  A fused-metrics
call then keeps its counters in the caller's workspace and still runs ONE kernel whose pixels, coefficients and sums
equal those of the ordinary path bit for bit; a round trip forced onto the TMA family takes the static tile split.

The capture pool belongs to the process, so these cases run in a child process: this file run as a script.  The child
inherits the test's environment (the arithmetic modes of the autouse fixture), prints its metrics and launch records
as JSON and leaves its pixels and coefficients in an .npz file."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import inputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

PATH_AUTO, PATH_TMA = 0, 2
ERR_ARG = -1
ZZ10 = "zz10"   # keep the first 10 zig-zag coefficients


def case_table():
    """name -> (pixels, keep, coefficient plane dtype or None, plan path, expected family)"""
    f = inputs.float_noise(1024, 2048, seed=3)
    u8 = np.random.default_rng(11).integers(0, 256, (256, 256), dtype=np.uint8)
    return {
        "u8": (u8, "all", None, PATH_AUTO, "direct"),
        "f32": (f, "all", None, PATH_AUTO, "direct"),
        "f32_i16": (f, "all", torch.int16, PATH_AUTO, "direct"),
        "f32_zz10": (f, ZZ10, None, PATH_AUTO, "direct"),
        "f32_zz10_i16": (f, ZZ10, torch.int16, PATH_AUTO, "direct"),
        "f32_tma": (f, "all", torch.float32, PATH_TMA, "tma"),
    }


class Call:
    """One b200dct_roundtrip_metrics call with its buffers, issued through the C ABI so that it can be captured."""

    def __init__(self, dct, img, keep, coef_dt, path):
        self.dct = dct
        mask = dct.ALL_COEFFS if keep == "all" else dct.api.zigzag_mask(10)
        self.plan = dct.Plan(keep=mask, path=path)
        self.x = torch.from_numpy(np.ascontiguousarray(img)).cuda()
        self.out = torch.empty_like(self.x)
        self.coef = None if coef_dt is None else torch.empty(img.shape, dtype=coef_dt, device="cuda")
        self.acc = torch.zeros(3, dtype=torch.float64, device="cuda")
        H, W = img.shape
        self.nbytes = int(dct.lib().b200dct_metrics_workspace_bytes(H, W))
        self.ws = torch.empty(max(1, self.nbytes // 8), dtype=torch.float64, device="cuda")

    def __call__(self, stream, nbytes=None):
        api = self.dct.api
        ip, idt, ipitch, H, W = api._plane(self.x)
        op, odt, opitch = api._plane(self.out)[:3]
        cp, cdt, cpitch = (None, api.F32, 0) if self.coef is None else api._plane(self.coef)[:3]
        return int(self.dct.lib().b200dct_roundtrip_metrics(
            self.plan._h, ip, idt, ipitch, op, odt, opitch, cp, cdt, cpitch, H, W, self.acc.data_ptr(), self.ws.data_ptr(),
            self.nbytes if nbytes is None else nbytes, api._stream(stream)))

    def sums(self):
        torch.cuda.synchronize()
        return self.acc.cpu().tolist()


def ordinary(dct, name):
    """(sse, energy, nnz) of the case made the ordinary way, on a scheduler slot"""
    c = Call(dct, *case_table()[name][:4])
    assert c(torch.cuda.current_stream()) == 0
    return c.sums()


def child_pool(dct, arrays):
    """Use the capture pool up, then capture each case once and replay it twice."""
    lib = dct.lib()
    s = torch.cuda.Stream()
    warm = Call(dct, np.zeros((64, 64), np.uint8), "all", None, PATH_AUTO)
    assert warm(s) == 0                                     # the first ordinary call creates the pools
    torch.cuda.synchronize()
    filler = torch.cuda.CUDAGraph()
    with torch.cuda.graph(filler, stream=s):
        for _ in range(int(lib.b200dct_capture_slots_left())):
            assert warm(s) == 0                             # a captured direct-family metrics call takes one slot
    res = {"slots_left_after_fill": int(lib.b200dct_capture_slots_left())}
    for name, (img, keep, coef_dt, path, _) in case_table().items():
        c = Call(dct, img, keep, coef_dt, path)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            rc = c(s)
            launches, family = dct.api.last_launch_count(), dct.api.last_path()
        g.replay()
        once = c.sums()
        arrays[name + "_out"] = c.out.cpu().numpy()
        if c.coef is not None:
            arrays[name + "_coef"] = c.coef.cpu().numpy()
        g.replay()
        res[name] = {"rc": rc, "launches": launches, "path": family, "once": once, "twice": c.sums(),
                     "slots_left": int(lib.b200dct_capture_slots_left())}
    # a round trip without metrics, forced onto the TMA family: without a ticket-counter pair, the static tile split
    x = torch.from_numpy(case_table()["f32_tma"][0]).cuda()
    out, coef = torch.empty_like(x), torch.empty_like(x)
    plan = dct.Plan(path=PATH_TMA)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        dct.roundtrip(x, out=out, coef=coef, plan=plan, stream=s)
        launches, family = dct.api.last_launch_count(), dct.api.last_path()
    for replay in (1, 2):
        out.fill_(float("nan"))
        coef.fill_(float("nan"))
        g.replay()
        torch.cuda.synchronize()
        arrays[f"plain{replay}_out"] = out.cpu().numpy()
        arrays[f"plain{replay}_coef"] = coef.cpu().numpy()
    res["plain"] = {"launches": launches, "path": family, "slots_left": int(lib.b200dct_capture_slots_left())}
    return res


def run_child(tmp_path):
    npz = tmp_path / "pool.npz"
    r = subprocess.run([sys.executable, os.path.abspath(__file__), str(npz)], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1]), np.load(npz)


def want(oracle, name):
    img, keep, coef_dt, _, _ = case_table()[name]
    kw = {} if keep == "all" else {"keep": oracle.zigzag_mask(10)}
    out, coef = oracle.roundtrip(img, want_coef=True, **kw)
    return out, (None if coef_dt is None else coef.astype(np.int16 if coef_dt == torch.int16 else np.float32))


def same_bits(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def test_metrics_with_the_capture_pool_used_up(dct, oracle, tmp_path):
    res, arrays = run_child(tmp_path)
    assert res["slots_left_after_fill"] == 0
    for name in case_table():
        r = res[name]
        assert r["rc"] == 0, name
        assert r["launches"] == 1 and r["path"] == case_table()[name][4], (name, r)
        assert r["slots_left"] == 0, name
        out, coef = want(oracle, name)
        assert same_bits(arrays[name + "_out"], out), name
        if coef is not None:
            assert same_bits(arrays[name + "_coef"], coef), name
        assert r["once"] == ordinary(dct, name), name           # the same bits as on a scheduler slot
        assert r["twice"] == [2 * v for v in r["once"]], name   # every replay adds the same sums
    # the static tile split: one launch on the TMA family, exact, and every replay the same
    r = res["plain"]
    assert r["launches"] == 1 and r["path"] == "tma" and r["slots_left"] == 0, r
    out, coef = want(oracle, "f32_tma")
    for replay in (1, 2):
        assert same_bits(arrays[f"plain{replay}_out"], out), replay
        assert same_bits(arrays[f"plain{replay}_coef"], coef), replay


def test_metrics_workspace_size(dct):
    c = Call(dct, np.zeros((64, 64), np.uint8), "all", None, PATH_AUTO)
    s = torch.cuda.current_stream()
    assert c(s, c.nbytes) == 0
    assert c(s, c.nbytes - 1) == ERR_ARG
    torch.cuda.synchronize()


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    import cuda_dct_idct_b200

    cuda_dct_idct_b200.lib()
    arrays = {}
    result = child_pool(cuda_dct_idct_b200, arrays)
    np.savez(sys.argv[1], **arrays)
    print(json.dumps(result))
