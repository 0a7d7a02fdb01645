"""pytest plugin: which of the libraries' kernels a test run launches.

    python -m pytest -m gpu -p tests.kernel_ledger_plugin [--kernel-ledger-out FILE] tests/
    PYTHONPATH=tests python -m pytest -m gpu -p kernel_ledger_plugin ...   (where another `tests` package
                                                                           on the path shadows this one)

Every test marked `gpu` runs under its own `torch.profiler` session (CUDA activity only); the kernel
names it records are mapped onto the inventory of the built libraries with the spelling of
tests/kernel_ledger.py.  At the end the plugin prints, and writes to FILE when given, the kernels that
were launched (with the first test that launched each), those that never were, and the tests that
started child processes: kernels launched only in a child are not seen by the profiler of this process.

Do not combine it with tests that run a profiler of their own (tests/test_gpu_kernel_matrix.py): only one
profiler session can be active in a process.
"""
from __future__ import annotations

import os
import subprocess
import sys
import time

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import kernel_ledger as KL  # noqa: E402


def _shown(arg, i) -> str:
    """A child's argument as the report shows it: the program by name, files of the repository relative to it,
    other absolute paths (temporary files) by name."""
    a = str(arg)
    if i == 0:
        return os.path.basename(a)
    if os.path.isabs(a):
        return os.path.relpath(a, KL.ROOT) if a.startswith(KL.ROOT + os.sep) else "<tmp>/" + os.path.basename(a)
    return a


def pytest_addoption(parser):
    parser.addoption("--kernel-ledger-out", default=None, help="write the kernel ledger report to this file")


class _Ledger:
    def __init__(self, out):
        self.out = out
        self.inv = None
        self.skip_reason = None
        self.first = {}        # key -> first test that launched it
        self.count = {}        # key -> tests that launched it
        self.raw = {}          # key -> one profiler spelling
        self.spawners = {}     # test -> argv of the child processes it started
        self.tests = 0
        self.outcomes = {"passed": 0, "failed": 0, "skipped": 0}

    def _ensure_inventory(self):
        if self.inv is None and self.skip_reason is None:
            if KL.tool("cuobjdump") is None or KL.tool("cu++filt") is None:
                self.skip_reason = "no cuobjdump / cu++filt in CUDA_HOME or on PATH"
            elif not KL.libraries_built():
                self.skip_reason = "the libraries are not built"
            else:
                self.inv = KL.inventory()
        return self.inv is not None

    @pytest.hookimpl(hookwrapper=True)
    def pytest_runtest_call(self, item):
        if item.get_closest_marker("gpu") is None or not self._ensure_inventory():
            yield
            return
        import torch
        from torch.profiler import ProfilerActivity, profile

        if not torch.cuda.is_available():
            yield
            return
        spawned = []
        orig = subprocess.Popen.__init__

        def popen(self_, args, *a, **kw):
            spawned.append(args if isinstance(args, str) else " ".join(_shown(x, i) for i, x in enumerate(args)))
            return orig(self_, args, *a, **kw)

        subprocess.Popen.__init__ = popen
        prof = profile(activities=[ProfilerActivity.CUDA])
        prof.__enter__()
        try:
            yield
        finally:
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
            prof.__exit__(None, None, None)
            subprocess.Popen.__init__ = orig
        self.tests += 1
        if spawned:
            self.spawners[item.nodeid] = spawned
        seen = set()
        for ev in prof.events():
            key = KL.canonical(ev.name)
            if key in self.inv and key not in seen:
                seen.add(key)
                self.raw.setdefault(key, ev.name)
                self.first.setdefault(key, item.nodeid)
                self.count[key] = self.count.get(key, 0) + 1

    def pytest_runtest_logreport(self, report):
        if report.when == "call" or (report.when == "setup" and report.outcome != "passed"):
            self.outcomes[report.outcome] = self.outcomes.get(report.outcome, 0) + 1

    def report_lines(self):
        if self.inv is None:
            return [f"kernel ledger: not recorded ({self.skip_reason or 'no GPU test ran'})"]
        launched = sorted(k for k in self.inv if k in self.first)
        never = sorted(k for k in self.inv if k not in self.first)
        lines = [f"kernel ledger: launched {len(launched)} of {len(self.inv)} kernels over {self.tests} GPU tests "
                 f"(outcomes: {self.outcomes})", "",
                 f"launched ({len(launched)}): key | tests that launched it | first test | profiler spelling"]
        lines += [f"  {k} | {self.count[k]} | {self.first[k]} | {self.raw[k]}" for k in launched]
        lines += ["", f"never launched in this process ({len(never)}): key | cu++filt spelling"]
        lines += [f"  {k} | {self.inv[k]}" for k in never]
        lines += ["", f"tests that started child processes ({len(self.spawners)}); kernels launched there are not recorded:"]
        for t, argv in sorted(self.spawners.items()):
            lines += [f"  {t}"] + [f"      {a}" for a in argv]
        return lines

    def pytest_terminal_summary(self, terminalreporter):
        lines = self.report_lines()
        for line in lines:
            terminalreporter.write_line(line)
        if self.out:
            gpu = "no GPU"
            try:
                import torch

                if torch.cuda.is_available():
                    gpu = torch.cuda.get_device_name(0)
            except Exception:
                pass
            with open(self.out, "w") as f:
                f.write(f"# {time.strftime('%Y-%m-%d')} on {gpu}: python -m pytest {' '.join(sys.argv[1:])}\n")
                f.write("\n".join(lines) + "\n")


def pytest_configure(config):
    config.pluginmanager.register(_Ledger(config.getoption("--kernel-ledger-out")), "kernel_ledger_recorder")
