"""CPU: the shape arithmetic and the trace parser of tests/tma_depth.py."""
import numpy as np
import pytest

import f64ref as R
import tma_depth as D


@pytest.mark.parametrize("sms", [1, 7, 132, 148, 160])
@pytest.mark.parametrize("warps", [8, 9, 12, 14, 16])
def test_deep_height_puts_every_warp_past_two_rounds(sms, warps):
    H = D.deep_height(sms, warps)
    S, n = sms * warps, D.ntiles(H, D.DEEP_W)
    assert H % 8 == 0
    assert n >= 3 * S + 1 and (n - 2 * S) % 2 == 1
    assert D.regime(n, sms, 32 * warps) == "R3"
    # the smallest such H: one block row less misses a condition
    m = D.ntiles(H - 8, D.DEEP_W)
    assert not (m >= 3 * S + 1 and (m - 2 * S) % 2 == 1)
    # and a grid of one CTA per SM: every CTA has more than `warps` tiles
    assert -(-n // warps) >= sms


@pytest.mark.parametrize("sms", [7, 132, 148])
@pytest.mark.parametrize("warps", [8, 9, 12, 14, 16])
def test_r2_height(sms, warps):
    H = D.r2_height(sms, warps)
    n = D.ntiles(H, D.DEEP_W)
    assert H % 8 == 0 and D.regime(n, sms, 32 * warps) == "R2"


def test_deep_width_ends_on_a_partial_tile():
    assert D.DEEP_W % 256 == 32 and D.tiles_x(D.DEEP_W) == 9
    assert D.ntiles(16, D.DEEP_W) == 18


def test_regimes():
    assert D.regime(100, 10, 320) == "R1" and D.regime(101, 10, 320) == "R2" and D.regime(200, 10, 320) == "R2"
    assert D.regime(301, 10, 320) == "R3" and D.regime(302, 10, 320) == "between" and D.regime(250, 10, 320) == "between"


def test_cta_warps():
    # f32 Haweel 8, dense 12, u8 16 (14 with an f32 plane), metrics 9
    assert D.cta_warps("f32", 1, ["f32", "f32"]) == 8
    assert D.cta_warps("f32", 2, ["f32", "f32", "i16"]) == 12
    assert D.cta_warps("u8", 1, ["u8", "u8"]) == 16
    assert D.cta_warps("u8", 1, ["u8", "u8", "i16"]) == 16
    assert D.cta_warps("u8", 0, ["u8", "u8", "f32"]) == 14
    assert D.cta_warps("u8", 1, ["f32", "u8"]) == 14
    assert D.cta_warps("f32", 1, ["f32", "f32"], metrics=True) == 9


def test_kernel_geometry():
    trace = {"traceEvents": [
        {"cat": "kernel", "name": "void b200dct::k_tma<2, 1, 0, 0, false, false>(b200dct::TmaParams)",
         "args": {"grid": [148, 1, 1], "block": [256, 1, 1]}},
        {"cat": "cuda_runtime", "name": "cudaLaunchKernel", "args": {}},
    ]}
    geo = D.kernel_geometry(trace)
    assert geo == [(trace["traceEvents"][0]["name"], (148, 1, 1), (256, 1, 1))]
    import kernel_ledger as KL
    assert D.tma_launch(geo, KL.canonical) == ("k_tma<2,1,0,0,0,0>", 148, 256)
    with pytest.raises(AssertionError, match="no grid / block"):
        D.kernel_geometry({"traceEvents": [{"cat": "kernel", "name": "k", "args": {"grid": [1, 1, 1]}}]})


def test_banded_checks_match_the_whole_image():
    rng = np.random.default_rng(3)
    H, W = 2 * D.BAND_ROWS + 16, 24
    img = rng.uniform(0, 255, (H, W)).astype(np.float32)
    T, Q = R.rand_sym_T(), np.full(64, 3.0, np.float32)
    Y, B = R.forward64(img, T)
    C = R.round_half_away(Y / R.tile(R.q_grid(Q), H, W)).astype(np.float32)
    whole = R.check_quant(C, Y, B, Q)
    banded = D.check_quant_banded(C, img, T, Q, R.ALL_COEFFS)
    assert banded.bad == whole.bad == 0 and banded.n == whole.n
    P, Bi = R.inverse64(C, T, Q)
    got = P.astype(np.float32)
    got[H - 3, 5] += 1.0      # one wrong pixel in the last band
    assert D.check_pixels_banded(got, C, T, Q).bad == R.check_close(got, P, Bi).bad == 1
