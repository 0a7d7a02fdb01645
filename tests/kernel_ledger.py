"""Which compiled kernels a test run launches: the inventory of the built libraries and one spelling of
kernel names that the inventory and the profiler share (numpy-free, no torch at import).

Inventory: every `__global__` entry of libb200dct.so and libb200dct_compat.so, read with `cuobjdump -elf`
of the toolkit that built them (one `.nv.info.<mangled name>` section per entry) and demangled with
`cu++filt`.  Recording: `torch.profiler` names a kernel with the C++ runtime's demangler.  The two
demanglers spell template arguments differently, so both go through `canonical()`:

    cu++filt:  void b200dct::k_direct<(int)2, (int)1, (int)0, (int)1, (bool)0, (bool)1>(b200dct::DirectParams)
    profiler:  void b200dct::k_direct<2, 1, 0, 1, false, true>(b200dct::DirectParams)
    canonical: k_direct<2,1,0,1,0,1>

A key keeps the unqualified kernel name and its template arguments, integers and bools as digits; the
return type, namespaces and parameter list go.  Names that are not kernels of the inventory (torch's
fills and copies, memsets) map to keys that are not in it and are filtered out by the caller.
"""
from __future__ import annotations

import os
import re
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "cuda-dct-idct_b200")
LIBRARIES = ("libb200dct.so", "libb200dct_compat.so")

_CAST = re.compile(r"\((?:int|bool|unsigned int|unsigned|long|unsigned long|char|unsigned char|short)\)\s*(?=-?\d)")
_ANON = re.compile(r"\(anonymous namespace\)::|<unnamed>::|\{anonymous\}::")
_WORDS = {"false": "0", "true": "1"}


def _top_level(s: str, i: int) -> bool:
    return s[:i].count("<") == s[:i].count(">")


def canonical(name: str) -> str:
    """One key per kernel, whichever demangler spelled `name` (see the module docstring)."""
    s = _ANON.sub("", name.strip())
    s = _CAST.sub("", s)
    # the parameter list: the first '(' outside the template argument list
    for i, ch in enumerate(s):
        if ch == "(" and _top_level(s, i):
            s = s[:i]
            break
    s = s.strip()
    # the return type: everything up to the last space outside the template argument list
    cut = -1
    for i, ch in enumerate(s):
        if ch == " " and _top_level(s, i):
            cut = i
    s = s[cut + 1:]
    # namespaces of the kernel itself (those of template arguments that are types stay)
    lt = s.find("<")
    head, args = (s, "") if lt < 0 else (s[:lt], s[lt:])
    head = head.rsplit("::", 1)[-1]
    if args:
        args = re.sub(r"\s*,\s*", ",", args)
        args = re.sub(r"\s*([<>])\s*", r"\1", args)
        args = re.sub(r"\b(false|true)\b", lambda m: _WORDS[m.group(1)], args)
    return head + args


def cuda_home() -> str:
    return os.environ.get("CUDA_HOME") or "/usr/local/cuda"


def tool(name: str) -> str | None:
    """A toolkit binary: $CUDA_HOME/bin first, then PATH; None if there is none."""
    p = os.path.join(cuda_home(), "bin", name)
    return p if os.access(p, os.X_OK) else shutil.which(name)


def mangled_entries(lib_path: str) -> list[str]:
    """Mangled names of the `__global__` entries of one shared library (cuobjdump -elf)."""
    out = subprocess.run([tool("cuobjdump"), "-elf", lib_path], capture_output=True, text=True, check=True).stdout
    return sorted(set(re.findall(r"CUDA_INFO\s.*\s\.nv\.info\.(_Z\S+)$", out, re.M)))


def demangle(mangled: list[str]) -> list[str]:
    if not mangled:
        return []
    out = subprocess.run([tool("cu++filt")], input="\n".join(mangled) + "\n", capture_output=True, text=True,
                         check=True).stdout
    names = out.splitlines()
    assert len(names) == len(mangled), "cu++filt returned a different number of names"
    return names


def inventory(lib_dir: str = PKG) -> dict[str, str]:
    """{canonical key: cu++filt name} of every kernel of the two libraries."""
    inv: dict[str, str] = {}
    for lib in LIBRARIES:
        for name in demangle(mangled_entries(os.path.join(lib_dir, lib))):
            key = canonical(name)
            assert key not in inv, f"two inventory entries share the key {key}: {inv[key]!r} and {name!r}"
            inv[key] = name
    return inv


def libraries_built(lib_dir: str = PKG) -> bool:
    return all(os.path.exists(os.path.join(lib_dir, lib)) for lib in LIBRARIES)
