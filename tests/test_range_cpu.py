"""CPU references for the wide-range contract: the baseline-JPEG coded size of zig-zag streams, in range
and out of it, and the oracle's int16 saturation of large coefficients.

The reference coder below is written from ITU-T T.81 alone (Annex C code lengths from the DHT
tables, F.1.2 categories, ZRL, EOB); it pins oracle_coded_bits, which the GPU suite then uses as the
reference of b200dct_zigzag_coded_bits."""
from __future__ import annotations

import numpy as np
import pytest

DC_MAX_CATEGORY = 11   # baseline: DC differences of magnitude <= 2047
AC_MAX_CATEGORY = 10   # baseline: AC values of magnitude <= 1023


def code_lengths(bits16, vals) -> dict:
    """T.81 Annex C: the BITS[l] symbols that follow in HUFFVAL order get codes of length l."""
    out, k = {}, 0
    for length in range(1, 17):
        for _ in range(int(bits16[length - 1])):
            out[int(vals[k])] = length
            k += 1
    return out


def reference_coded_bits(stream, table, oracle):
    """(bits of the in-range symbols, whether any symbol lies outside the baseline categories)."""
    dcl = code_lengths(*oracle.huffman_spec(0, table))
    acl = code_lengths(*oracle.huffman_spec(1, table))
    bits, out_of_range, prev = 0, False, 0
    for blk in np.asarray(stream).reshape(-1, 64).astype(int):
        d = int(blk[0]) - prev
        prev = int(blk[0])
        s = abs(d).bit_length()
        if s <= DC_MAX_CATEGORY:
            bits += dcl[s] + s
        else:
            out_of_range = True
        run = 0
        for v in blk[1:]:
            v = int(v)
            if v == 0:
                run += 1
                continue
            while run > 15:
                bits += acl[0xF0]
                run -= 16
            s = abs(v).bit_length()
            if s <= AC_MAX_CATEGORY:
                bits += acl[(run << 4) | s] + s
            else:
                out_of_range = True
            run = 0
        if run:
            bits += acl[0x00]
    return bits, out_of_range


def in_range_stream(nblk, seed):
    """Random block-major zig-zag streams that reach every baseline extreme: AC +-1023, DC steps of
    +-2047, runs of more than 16 zeros (ZRL), blocks that end in zeros (EOB) and blocks that do not."""
    rng = np.random.default_rng(seed)
    s = np.zeros((nblk, 64), np.int32)
    for b in range(nblk):
        kind = b % 4
        nz = rng.integers(0, 64) if kind else 63
        pos = rng.choice(np.arange(1, 64), size=nz, replace=False)
        s[b, pos] = rng.choice([-1023, 1023, -1, 1, -512, 511, 3], size=nz) if kind != 2 else rng.integers(-1023, 1024, size=nz)
        if kind == 3:
            s[b, 63] = 1023          # a value after a long run: ZRLs, no EOB
    # DC walks that take steps of exactly +-2047 (and stay within int16)
    dc = 0
    for b, step in enumerate(rng.choice([-2047, 2047, 0, 5], size=nblk)):
        dc += -step if abs(dc + step) > 30000 else step
        s[b, 0] = dc
    return s.astype(np.int16)


@pytest.mark.parametrize("table", [0, 1])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_coded_bits_matches_reference_in_range(oracle, table, seed):
    s = in_range_stream(96, seed)
    assert np.abs(s[:, 1:]).max() == 1023
    assert np.abs(np.diff(np.concatenate([[0], s[:, 0].astype(int)]))).max() == 2047
    want, flag = reference_coded_bits(s, table, oracle)
    assert not flag
    assert oracle.coded_bits(s, table) == want


@pytest.mark.parametrize("table", [0, 1])
def test_oracle_coded_bits_on_real_streams(oracle, table):
    img = oracle.rand_image(64, 64, 5)
    for Q in (oracle.jpeg_Q(), np.ones(64, np.float32), oracle.jpeg_Q() / 4):
        s = oracle.zigzag_i16(oracle.dct(img, Q=Q))
        want, flag = reference_coded_bits(s, table, oracle)
        assert oracle.coded_bits(s, table) == want | (flag << 63)


def out_of_range_cases():
    """(name, stream): each holds exactly one kind of symbol that baseline JPEG cannot code."""
    cases = []
    s = np.zeros((4, 64), np.int16)
    s[1, 5] = 1024
    cases.append(("AC +1024", s))
    s = np.zeros((4, 64), np.int16)
    s[2, 63] = -1024
    cases.append(("AC -1024", s))
    s = np.zeros((4, 64), np.int16)
    s[1, 0] = 2048
    cases.append(("DC step +2048", s))
    s = np.zeros((4, 64), np.int16)
    s[0, 0], s[1, 0] = 100, 100 - 2048
    cases.append(("DC step -2048", s))
    s = np.zeros((4, 64), np.int16)
    s[1, 0], s[2, 0] = 32767, -32768       # a DC difference of -65535: category 16
    cases.append(("DC 32767 then -32768", s))
    s = np.zeros((4, 64), np.int16)
    s[3, 16] = -32768                      # 15 zeros, then category 16: run/size 0xF0 | 16 lies past the table
    cases.append(("-32768 after 15 zeros", s))
    return cases


@pytest.mark.parametrize("table", [0, 1])
@pytest.mark.parametrize("case", range(6))
def test_oracle_flags_symbols_outside_the_baseline_categories(oracle, table, case):
    name, s = out_of_range_cases()[case]
    want, flag = reference_coded_bits(s, table, oracle)
    assert flag, name
    got = oracle.coded_bits(s, table)
    assert got >> 63 == 1, name
    assert got & ((1 << 63) - 1) == want, name     # the in-range symbols are still counted
    with pytest.raises(ValueError):
        oracle.compression_factor(oracle.unzigzag_i16(s.reshape(1, 4, 64)), table)


def test_sub_unit_quantisers_leave_the_baseline_range(oracle):
    """Every Q entry 1/16 (the RGB split's documented floor) on random 8-bit content already yields
    AC values above 1023: the coded size has to say so rather than count them as 0 bits."""
    img = oracle.rand_image(64, 64, 3)
    coef = oracle.dct(img, Q=np.full(64, 1 / 16, np.float32))
    assert (np.abs(coef.reshape(8, 8, 8, 8).transpose(0, 2, 1, 3).reshape(-1, 64)[:, 1:]) > 1023).sum() > 100
    assert oracle.coded_bits(oracle.zigzag_i16(coef), 0) >> 63 == 1


def test_oracle_zigzag_saturates_like_clip(oracle):
    """oracle.zigzag_i16 is the rule every saturating coefficient writer is held to: round, then clip."""
    rng = np.random.default_rng(4)
    img = (rng.random((32, 32)) * 2e6 - 1e6).astype(np.float32)
    coef = oracle.dct(img)
    assert np.abs(coef).max() > 40000
    zz = oracle.zigzag_i16(coef)
    back = oracle.unzigzag_i16(zz)
    assert np.array_equal(back, np.clip(coef, -32768, 32767))
