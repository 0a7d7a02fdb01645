"""CPU: the one spelling of kernel names that the kernel ledger (tests/kernel_ledger.py) gives the inventory
of the built libraries (cu++filt) and the profiler's records (the C++ runtime's demangler)."""
from __future__ import annotations

import pytest

import kernel_ledger as KL

# (torch.profiler spelling, cu++filt spelling, key): one per kernel template.  The profiler names are
# copied from a torch.profiler record of the kernel on a B200 (torch 2.11, CUDA 12.8 runtime).
PAIRS = [
    ("void b200dct::k_direct<2, 1, 0, 1, false, true>(b200dct::DirectParams)",
     "void b200dct::k_direct<(int)2, (int)1, (int)0, (int)1, (bool)0, (bool)1>(b200dct::DirectParams)",
     "k_direct<2,1,0,1,0,1>"),
    ("void b200dct::k_tma<2, 1, 2, 1, true, false>(b200dct::TmaParams)",
     "void b200dct::k_tma<(int)2, (int)1, (int)2, (int)1, (bool)1, (bool)0>(b200dct::TmaParams)",
     "k_tma<2,1,2,1,1,0>"),
    ("void b200dct::k_any<0, 1, 0, false>(b200dct::AnyParams)",
     "void b200dct::k_any<(int)0, (int)1, (int)0, (bool)0>(b200dct::AnyParams)",
     "k_any<0,1,0,0>"),
    ("void b200dct::k_any_u8<1, 2, true>(b200dct::AnyParams)",
     "void b200dct::k_any_u8<(int)1, (int)2, (bool)1>(b200dct::AnyParams)",
     "k_any_u8<1,2,1>"),
    ("void b200dct::k_rgb<2, true, false>(b200dct::RgbParams)",
     "void b200dct::k_rgb<(int)2, (bool)1, (bool)0>(b200dct::RgbParams)",
     "k_rgb<2,1,0>"),
    ("void b200dct::k_rgb_forward<1>(b200dct::RgbParams)",
     "void b200dct::k_rgb_forward<(int)1>(b200dct::RgbParams)",
     "k_rgb_forward<1>"),
    ("void b200dct::k_rgb_inverse<true>(b200dct::RgbParams)",
     "void b200dct::k_rgb_inverse<(bool)1>(b200dct::RgbParams)",
     "k_rgb_inverse<1>"),
    ("void b200dct::k_rgb420_forward<2>(b200dct::Rgb420Params)",
     "void b200dct::k_rgb420_forward<(int)2>(b200dct::Rgb420Params)",
     "k_rgb420_forward<2>"),
    ("void b200dct::k_rgb420_inverse<false>(b200dct::Rgb420Params)",
     "void b200dct::k_rgb420_inverse<(bool)0>(b200dct::Rgb420Params)",
     "k_rgb420_inverse<0>"),
    ("void b200dct::k_mma<true>(b200dct::MmaParams)",
     "void b200dct::k_mma<(bool)1>(b200dct::MmaParams)",
     "k_mma<1>"),
    ("void k_metrics<unsigned char>(unsigned char const*, unsigned char const*, unsigned long, int, int, double*)",
     "void k_metrics<unsigned char>(const T1 *, const T1 *, unsigned long, int, int, double *)",
     "k_metrics<unsigned char>"),
    ("k_coded_bits((anonymous namespace)::CodedParams)",
     "k_coded_bits(<unnamed>::CodedParams)",
     "k_coded_bits"),
    ("k_selftest_div(float, unsigned long long, unsigned long long, unsigned long long*)",
     "k_selftest_div(float, unsigned long long, unsigned long long, unsigned long long *)",
     "k_selftest_div"),
    ("(anonymous namespace)::k_dequant_inplace(float*, float const*, int, unsigned long)",
     "<unnamed>::k_dequant_inplace(float *, const float *, int, unsigned long)",
     "k_dequant_inplace"),
]


@pytest.mark.parametrize("prof,filt,key", PAIRS, ids=[p[2] for p in PAIRS])
def test_both_spellings_map_to_one_key(prof, filt, key):
    assert KL.canonical(prof) == key
    assert KL.canonical(filt) == key


def test_keys_separate_what_differs():
    """Every template argument is part of the key: two kernels that differ in one argument never share it."""
    base = "void b200dct::k_direct<(int)2, (int)1, (int)0, (int)1, (bool)0, (bool)0>(b200dct::DirectParams)"
    args = ["(int)2", "(int)1", "(int)0", "(int)1", "(bool)0", "(bool)0"]
    keys = {KL.canonical(base)}
    for i, a in enumerate(args):
        other = list(args)
        other[i] = "(bool)1" if a.startswith("(bool)") else f"(int){int(a[5:]) + 1}"
        keys.add(KL.canonical(f"void b200dct::k_direct<{', '.join(other)}>(b200dct::DirectParams)"))
    assert len(keys) == 1 + len(args)
    assert KL.canonical("void k_metrics<float>(const T1 *)") != KL.canonical("void k_metrics<unsigned char>(const T1 *)")
    assert KL.canonical("void b200dct::k_tma<2, 1, 0, 0, false, false>(b200dct::TmaParams)") != \
        KL.canonical("void b200dct::k_direct<2, 1, 0, 0, false, false>(b200dct::DirectParams)")


def test_foreign_kernels_do_not_collide():
    """torch's own kernels and memsets, as the profiler names them, map to keys outside the library's."""
    for name in ("void at::native::vectorized_elementwise_kernel<4, at::native::FillFunctor<float>, "
                 "std::array<char*, 1ul> >(int, at::native::FillFunctor<float>, std::array<char*, 1ul>)",
                 "Memset (Device)", "Memcpy HtoD (Pageable -> Device)"):
        key = KL.canonical(name)
        assert not key.startswith(("k_direct", "k_tma", "k_any", "k_rgb", "k_mma", "k_metrics", "k_coded", "k_selftest"))


needs_tools = pytest.mark.skipif(KL.tool("cuobjdump") is None or KL.tool("cu++filt") is None,
                                 reason="no cuobjdump / cu++filt in CUDA_HOME or on PATH")
needs_libs = pytest.mark.skipif(not KL.libraries_built(), reason="the libraries are not built")


@needs_tools
def test_cufilt_spelling_of_the_fixed_names():
    """cu++filt itself produces the inventory spellings above from the mangled names."""
    mangled = ["_ZN7b200dct8k_directILi2ELi1ELi0ELi1ELb0ELb1EEEvNS_12DirectParamsE",
               "_ZN7b200dct5k_tmaILi2ELi1ELi2ELi1ELb1ELb0EEEvNS_9TmaParamsE",
               "_Z9k_metricsIhEvPKT_S2_miiPd"]
    got = KL.demangle(mangled)
    assert [KL.canonical(g) for g in got] == ["k_direct<2,1,0,1,0,1>", "k_tma<2,1,2,1,1,0>", "k_metrics<unsigned char>"]


@needs_tools
@needs_libs
def test_inventory_keys_are_distinct():
    """Every entry of the built libraries maps to a key of its own (inventory() asserts it while building
    the map), and the map holds every entry: 181 kernels in libb200dct.so and one in the compat library."""
    inv = KL.inventory()
    n = sum(len(KL.mangled_entries(f"{KL.PKG}/{lib}")) for lib in KL.LIBRARIES)
    assert len(inv) == n
    assert len(KL.mangled_entries(f"{KL.PKG}/libb200dct_compat.so")) == 1
    for name in inv.values():
        assert KL.canonical(name) in inv
