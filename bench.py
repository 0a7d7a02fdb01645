#!/usr/bin/env python
"""bench.py -- Gpixel/s of the fused DCT -> quantise -> IDCT hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-gpu]
                    [--dump-outputs DIR]

One "step" = one fused pass (b200dct_roundtrip, HpApprDCT: Haweel T, JPEG Q, all
coefficients kept) over one 8192 x 8192 fp32 image per GPU -- BASELINE.json configs[1].
For N > 1 (launched with torchrun, one rank per GPU) every rank owns one 8192-row stripe
of an (N*8192) x 8192 image: block-row striping, no halo, no data-path collective, weak
scaling.  Rank 0 prints ONE JSON line.

Legs of the default arm, all on the same workload:
  value        device-resident: inputs already in HBM, exactly K launches timed with CUDA
               events on the launching stream, barrier + synchronize on both sides, max over ranks;
               the step rotates over 4 input/output buffer pairs (2 GiB) so nothing is L2
               resident (one image pair alone is 512 MiB against a 126 MB L2).
  roofline     algorithmic bytes per launch (8 B/px: 4 read + 4 written) / average launch
               time from the same events, against the measured HBM copy peak
               (MEASURED_PEAKS.json, else the profiling guide's fallback).
  e2e          the same metric through the host-buffer entry point
               (b200dct_roundtrip_host): pinned host image in, pinned host image out, H2D
               and D2H inside the timed region, every step.
  cpu_baseline the sequential CPU restatement of the reference (oracle/, 1 thread) on the
               whole 8192^2 image, rank 0 / N=1 only.  A reported baseline, not the target.
  reference_gpu the UNMODIFIED reference kernels (oracle/_ref, HpApprDCT recompiled for
               sm_100a) on the same device buffers: its own printed event times.

--impl reference: the reference arm of the contract.  The reference ships no CPU code
(SURVEY.md S1), so this is the oracle port on all host threads, rank 0 only.
--impl reference-gpu: the unmodified reference GPU program flow (host image -> H2D ->
dct_all_blocks_cuda -> idct_all_blocks_cuda -> D2H) from oracle/_ref, for context.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_SIDE = 8192
METRIC = "Gpixel/s DCT+quant+IDCT at 8192^2 fp32 (HpApprDCT fused round trip)"
UNIT = "Gpixel/s"
BYTES_PER_PX = 8.0  # algorithmic: 4 B read + 4 B written per pixel (SURVEY.md section 8d)


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU while the timed region runs
    (NVML, the same counters `nvidia-smi --query-gpu=clocks.sm,...` prints)."""

    def __init__(self, index: int, period_s: float = 0.02):
        self.index, self.period = index, period_s
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        self._nvml = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None
            return self
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def _run(self):
        nv = self._nvml
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=2)
        d = {"sm_mhz": (statistics.median(self.samples) if self.samples else None),
             "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}
        return d


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the headline kernel from the
    committed ncu capture (profiles/*traffic.json), or None."""
    try:
        best = None
        pd = os.path.join(ROOT, "profiles")
        for f in sorted(os.listdir(pd)):
            if f.endswith("traffic.json"):
                with open(os.path.join(pd, f)) as fh:
                    best = json.load(fh)
        return None if best is None else float(best["dram_bytes_per_launch"])
    except Exception:
        return None


# ------------------------------------------------------------------ reference arms
def run_reference_cpu(args):
    """Contract's reference arm: CPU, host cores only, rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import numpy as np

    from oracle import oracle as o

    o.build()
    rows = 2048                                     # bounded sample: a 2048-row stripe of the 8192^2 image
    img = o.rand_image(rows, N_SIDE, 42)
    threads_all = max(1, len(os.sched_getaffinity(0)))
    # pick the thread count that is actually faster on this box (containers often cap CPU time)
    t1 = o.time_roundtrip(img, reps=1, threads=1)
    tn = o.time_roundtrip(img, reps=1, threads=threads_all) if threads_all > 1 else t1
    threads = threads_all if tn < t1 else 1
    # keep the whole run bounded (~90 s) whatever K the driver passes: shrink the stripe
    per_step = min(t1, tn)
    budget = 90.0 / max(1, args.steps + args.warmup)
    if per_step > budget:
        rows = max(64, int(rows * budget / per_step) // 8 * 8)
        img = np.ascontiguousarray(img[:rows])
    out = np.empty_like(img)
    for _ in range(args.warmup):
        o.time_roundtrip(img, reps=1, threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o.lib().oracle_roundtrip(img, rows, N_SIDE, o.haweel_T(), o.jpeg_Q(), o.ALL_COEFFS, None, out, threads)
    dt = time.perf_counter() - t0
    gpx = rows * N_SIDE * args.steps / dt / 1e9
    sample = f"{rows}x{N_SIDE} f32 stripe of the 8192^2 image per step, srand(42) rand()%256"
    line = {
        "impl": "reference", "metric": METRIC, "value": gpx, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "8192x8192 fp32 HpApprDCT DCT+quant+IDCT (BASELINE configs[1]); CPU sample: " + sample,
                   "note": "the reference ships no CPU implementation (SURVEY.md S1); this is the oracle port of its "
                           "arithmetic (oracle/dct_oracle.c, gcc -O2, OpenMP over block-rows)"},
        "cpu_baseline": {"value": gpx, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "t_1thread_s": t1, "t_allthreads_s": tn, "host_threads_available": threads_all},
        "e2e": {"value": gpx, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "extrapolation": "each step transforms a stripe of the 8192^2 image, not the whole image; the rate is per pixel and "
                         "8x8 blocks are independent, so it is size-independent (same arithmetic per block at any H)",
    }
    print(json.dumps(line))
    return 0


def run_reference_gpu(args):
    """The unmodified reference GPU flow, for context (not the contract's reference arm)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import refgpu
    from oracle import oracle as o

    if not refgpu.available("newappr") or not torch.cuda.is_available():
        print(json.dumps({"impl": "reference-gpu", "unavailable": "oracle/_ref/libref_newappr.so not built or no GPU"}))
        return 0
    torch.cuda.set_device(0)
    refgpu.set_quant("newappr", o.jpeg_Q())
    T = torch.from_numpy(o.haweel_T()).cuda()
    h_img = torch.randint(0, 256, (N_SIDE, N_SIDE), dtype=torch.int32).float().pin_memory()
    h_out = torch.empty_like(h_img).pin_memory()
    d_img, d_coef, d_rec = (torch.empty(N_SIDE, N_SIDE, device="cuda") for _ in range(3))
    kms = []

    def step():
        d_img.copy_(h_img, non_blocking=True)
        _, t1 = refgpu.dct("newappr", d_img, T, d_coef)
        _, t2 = refgpu.idct("newappr", d_coef, T, d_rec)
        h_out.copy_(d_rec, non_blocking=True)
        torch.cuda.synchronize()
        kms.append(t1 + t2)

    for _ in range(args.warmup):
        step()
    kms.clear()
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    px = N_SIDE * N_SIDE
    line = {
        "impl": "reference-gpu", "metric": METRIC, "value": px * steps / dt / 1e9, "unit": UNIT, "n_gpus": 1,
        "steps": steps, "warmup": args.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "8192x8192 fp32, reference main() flow: pinned host -> H2D -> dct_all_blocks_cuda -> "
                               "idct_all_blocks_cuda -> D2H (main_newAppr.cu:88-124), HpApprDCT recompiled for sm_100a"},
        "kernel_only": {"ms": statistics.mean(kms), "gpixel_s": px / (statistics.mean(kms) * 1e-3) / 1e9,
                        "what": "sum of the reference's own printed DCT and IDCT event times (6 launches, 48 B/px)"},
        "e2e": {"value": px * steps / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": px * 4, "d2h_bytes_per_step": px * 4},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------ our arm
WINDOWS = 5   # the K timed steps are split into up to 5 consecutive windows; the median window is reported
DUMP_ROWS = 1024   # --dump-outputs: rows of output written in all, shared by the ranks (32 MiB of f32)


def split_steps(k, windows=WINDOWS):
    """Window sizes that add up to exactly k steps (at most `windows` windows, sizes differ by <= 1)."""
    n = max(1, min(windows, k))
    return [k // n + (1 if w < k % n else 0) for w in range(n)]


def timed_windows(step, sizes, stream, warm=0):
    """Enqueue `warm` untimed steps and then one window of sizes[w] steps per entry on `stream`, with
    NO host synchronisation anywhere in between: event i sits between window i-1 and window i, so
    every window starts on a busy GPU (the first launch of a window overlaps the previous kernel's
    tail exactly like every other launch).  Returns the window times in ms."""
    import torch

    evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(sizes) + 1)]
    for i in range(warm):
        step(i)
    evs[0].record(stream)
    n = warm
    for w, k in enumerate(sizes):
        for _ in range(k):
            step(n)
            n += 1
        evs[w + 1].record(stream)
    torch.cuda.synchronize()
    return [evs[w].elapsed_time(evs[w + 1]) for w in range(len(sizes))]


def rotating(m, plan, ins, outs, stream, coef=None):
    def step(i):
        m.roundtrip(ins[i % len(ins)], out=outs[i % len(outs)], coef=coef, plan=plan, stream=stream)
    return step


def run_ours(args):
    import numpy as np
    import torch

    import cuda_dct_idct_b200 as m

    rank, local_rank, world = m.dist.init()
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    m.lib()
    plan = m.Plan()
    px = N_SIDE * N_SIDE                       # pixels per rank per step
    H0, H1 = m.stripe_rows(N_SIDE * world, world, rank)   # this rank's stripe of the (N*8192) x 8192 image
    assert H1 - H0 == N_SIDE
    K, W = args.steps, max(args.warmup, 3)

    # ---- device-resident leg: 4 rotating buffer pairs, synthetic integers 0..255
    NBUF = 4
    g = torch.Generator(device=dev).manual_seed(42 + rank)
    ins = [torch.randint(0, 256, (N_SIDE, N_SIDE), device=dev, generator=g, dtype=torch.int32).float() for _ in range(NBUF)]
    outs = [torch.empty(N_SIDE, N_SIDE, device=dev) for _ in range(NBUF)]
    stream = torch.cuda.current_stream()
    launches = 0

    def step(i):
        nonlocal launches
        m.roundtrip(ins[i % NBUF], out=outs[i % NBUF], plan=plan, stream=stream)
        launches += m.api.last_launch_count()

    step(0)
    torch.cuda.synchronize()
    kernel_path = m.api.last_path()

    # Timed region.  barrier + synchronize, then W warm-up steps and exactly K timed steps, split
    # into up to WINDOWS consecutive windows, are enqueued back to back with no synchronisation in
    # between; barrier + synchronize after.  Reported: the MEDIAN window's time per step (per
    # rank), max over ranks.
    sizes = split_steps(K)
    sampler = ClockSampler(local_rank).start()
    m.dist.barrier()
    torch.cuda.synchronize()
    launches = 0
    windows = timed_windows(step, sizes, stream, warm=W)
    m.dist.barrier()
    timed_launches = launches - W                     # kernels launched inside the timed windows
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs[(W + K - 1) % NBUF], rank, world)   # what the last timed step returned
    ms_local = statistics.median(ms / k for ms, k in zip(windows, sizes))   # per step
    # keep the identical load running briefly if the timed region was too short to sample clocks
    extra = 0
    t_end = time.perf_counter() + (0.0 if sum(windows) > 400 else 0.6)
    while time.perf_counter() < t_end:
        for i in range(64):
            m.roundtrip(ins[i % NBUF], out=outs[i % NBUF], plan=plan, stream=stream)
        torch.cuda.synchronize()
        extra += 64
    clocks = sampler.stop()
    clocks["sampled_over"] = "timed region" if extra == 0 else f"timed region + {extra} identical launches (region < 0.4 s)"
    ms_per_step = m.dist.max_over_ranks(ms_local, dev)
    per_rank = m.dist.all_ranks(ms_local, dev)
    first_window = m.dist.max_over_ranks(windows[0] / sizes[0], dev)
    value = px * world / (ms_per_step * 1e-3) / 1e9

    # per-launch duration of the dominant kernel: a window is nothing but back-to-back launches
    # of it on this stream, so window time / its steps is its average duration
    peak, peak_src = measured_peak()
    k_ms = ms_local
    achieved = BYTES_PER_PX * px / (k_ms * 1e-3) / 1e9
    traffic = ncu_traffic()
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": "committed ncu --set full capture (profiles/*traffic.json), not measured in this run",
                "peak_source": peak_src, "kernel": f"k_{kernel_path}<RT,sparse,Q_IMM,f32>",
                "algorithmic_bytes_per_launch": BYTES_PER_PX * px, "avg_launch_ms": k_ms,
                "frac_of_nominal_8TBs": achieved / 8000.0,
                "frac_note": "frac can exceed 1: the denominator is a measured copy-kernel peak, and a copy kernel pays a read-only ramp and a "
                             "write-only tail at its launch boundaries, which consecutive launches of this kernel overlap (early tile loads, DESIGN.md section 4)"}

    # ---- parity on EVERY rank: bands of what was just computed against the oracle (bit-exact)
    parity_local = True
    try:
        from oracle import oracle as o

        for b, r0 in ((0, 0), (0, N_SIDE - 16), (1 % NBUF, N_SIDE // 2 + 8)):
            band = ins[b][r0:r0 + 16].cpu().numpy()
            parity_local = parity_local and bool(np.array_equal(outs[b][r0:r0 + 16].cpu().numpy().view(np.uint32),
                                                                o.roundtrip(band).view(np.uint32)))
    except Exception as e:  # pragma: no cover
        parity_local = False
        print(f"rank {rank}: parity check failed to run: {e}", file=sys.stderr)
    parity_all = m.dist.sum_over_ranks(0.0 if parity_local else 1.0, dev) == 0.0

    # ---- e2e leg
    e2e = e2e_leg(m, plan, dev, world, args)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"{N_SIDE}x{N_SIDE} fp32 image per GPU, HpApprDCT (Haweel T, JPEG luminance Q, 64 coefficients kept), "
                               "fused DCT+quant+dequant+IDCT (BASELINE configs[1])",
                   "striping": f"{world} block-row stripe(s) of a {N_SIDE * world}x{N_SIDE} image, no halo, no collective",
                   "l2": "inputs larger than L2: 4 rotating in/out pairs, 2 GiB working set vs 126 MB L2",
                   "timing": f"barrier+synchronize, then {W} warm-up steps and exactly {K} timed steps in {len(sizes)} consecutive "
                             f"windows of {'/'.join(map(str, sizes))} steps enqueued back to back on one stream (CUDA events between "
                             "windows, no host synchronisation inside), barrier+synchronize; ms_per_step = median over windows of "
                             "window time / its steps, max over ranks",
                   "launch": "consecutive launches overlap tail and set-up through programmatic dependent launch "
                             "(each kernel waits for its predecessor before touching memory)",
                   "kernel_path": kernel_path},
        "windows_ms": windows, "window_steps": sizes, "first_window_ms_per_step": first_window,
        "per_rank_ms_per_step": {"min": min(per_rank), "median": statistics.median(per_rank), "max": max(per_rank),
                                 "all": per_rank},
        "roofline": roofline, "e2e": e2e, "gpu_launches": timed_launches, "clocks": clocks,
        "parity_all_ranks": bool(parity_all),
        "parity_check": "every rank: 3 bands (48 rows) of its timed output against the CPU oracle, bit-exact; all-reduced",
    }

    # ---- the other BASELINE configs, outside the timed value (each its own small timed loop)
    del ins, outs
    torch.cuda.empty_cache()
    try:
        if world == 1:
            line["extras"] = extras_single_gpu(m, dev, peak)
        else:
            line["extras"] = extras_multi_gpu(m, dev, rank, world)
    except Exception as e:  # pragma: no cover
        line["extras"] = {"error": repr(e)}

    # ---- baselines, rank 0 at N=1 only
    if rank == 0 and world == 1 and not args.no_baselines:
        line["cpu_baseline"] = cpu_baseline()
        a = torch.randint(0, 256, (N_SIDE, N_SIDE), device=dev, dtype=torch.int32).float()
        ref = reference_gpu_kernels(a, torch.empty_like(a))
        if ref:
            line["reference_gpu"] = ref
    if rank == 0:
        print(json.dumps(line))
    m.dist.barrier()
    m.dist.shutdown()
    return 0


def dump_outputs(out_dir, out, rank, world):
    """Write DUMP_ROWS // world rows of this rank's output image `out` (a fixed, seeded choice of
    rows, the same in every run) to out_dir/out_rank<rank>.npy as float32: DUMP_ROWS rows, 32 MiB,
    over all ranks."""
    import numpy as np
    import torch

    rows = np.sort(np.random.default_rng(0).choice(out.shape[0], max(1, DUMP_ROWS // world), replace=False))
    sample = out.index_select(0, torch.from_numpy(rows).to(out.device)).float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"out_rank{rank}.npy"), sample)


def e2e_leg(m, plan, dev, world, args):
    """The same metric through the host-buffer entry point: pinned host image in, pinned host image
    out, H2D and D2H inside the timed region, every step."""
    import torch

    px = N_SIDE * N_SIDE
    e2e_steps = max(3, min(args.steps, 20))
    res = {}
    for name, dtype, es in (("f32", torch.float32, 4), ("u8", torch.uint8, 1)):
        h_in = torch.randint(0, 256, (N_SIDE, N_SIDE), dtype=torch.int32).to(dtype).pin_memory()
        h_outs = [torch.empty(N_SIDE, N_SIDE, dtype=dtype).pin_memory() for _ in range(2)]
        # the pipeline is a long-lived object of the caller (streams + chunk buffers): created and
        # warmed up before the timed region, closed after it
        pipe = m.HostPipeline(plan=plan)
        for i in range(2):
            pipe.submit(h_in, h_outs[i % 2])
        pipe.drain()
        m.dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        # consecutive images overlap: image i+1 is being uploaded while image i is still on its way back
        for i in range(e2e_steps):
            pipe.submit(h_in, h_outs[i % 2])
        pipe.drain()                                     # every h_out complete in host memory
        api = ("b200dct_host_pipeline_submit/_drain (pinned host in/out, chunked H2D/kernel/D2H pipeline, "
               f"{pipe.chunk_bytes >> 20} MiB chunks, consecutive images overlap)")
        torch.cuda.synchronize()
        local = time.perf_counter() - t0
        m.dist.barrier()
        secs = m.dist.max_over_ranks(local, dev)
        pipe.close()
        # latency of ONE image through the synchronous one-call form (pays a fill/drain bubble per call)
        m.roundtrip_host(h_in, h_outs[0], plan=plan)
        t1 = time.perf_counter()
        for i in range(3):
            m.roundtrip_host(h_in, h_outs[i % 2], plan=plan)
        sync_ms = (time.perf_counter() - t1) / 3 * 1e3
        res[name] = {"single_image_sync_call_ms": sync_ms, "value": px * world * e2e_steps / secs / 1e9, "unit": UNIT, "h2d_bytes_per_step": px * es * world,
                     "d2h_bytes_per_step": px * es * world, "steps": e2e_steps, "ms_per_step": secs / e2e_steps * 1e3,
                     "api": api, "host_gb_s_each_way": px * es * world * e2e_steps / secs / 1e9}
        del h_in, h_outs
    e2e = res["f32"]
    ceil = pcie_ceiling(world)
    if ceil:
        e2e["pcie_ceiling_gb_s_each_way"] = ceil["gb_s_each_way"]
        e2e["pcie_ceiling_source"] = ceil["source"]
        e2e["frac_of_pcie_ceiling"] = e2e["host_gb_s_each_way"] / ceil["gb_s_each_way"]
    e2e["u8"] = res["u8"]    # the reference's file-level data is 8-bit (utils.cu:10-15): 4x fewer PCIe bytes
    return e2e


def pcie_ceiling(world):
    """Copies-only duplex host<->device ceiling for `world` ranks of this pool, measured by
    benchmarks/experiments/pcie.py under torchrun and committed as profiles/*pcie_ceiling.json."""
    try:
        pd = os.path.join(ROOT, "profiles")
        best = None
        for f in sorted(os.listdir(pd)):
            if f.endswith("pcie_ceiling.json"):
                with open(os.path.join(pd, f)) as fh:
                    best = json.load(fh)
        row = best["ranks"][str(world)]
        return {"gb_s_each_way": float(row["duplex_gb_s_each_way_aggregate"]), "source": best["source"]}
    except Exception:
        return None


def time_config(m, step, k=20, windows=3, warm=5):
    import torch

    w = timed_windows(step, [k] * windows, torch.cuda.current_stream(), warm=warm)
    return statistics.median(w) / k


def extras_single_gpu(m, dev, peak):
    """BASELINE configs[2..3] and the u8 dtype of configs[4] on one GPU; every number is device time
    per pass (median of 3 windows of 20 back-to-back passes, rotating buffers larger than L2)."""
    import torch

    from oracle import oracle as o   # only for the DCT-II matrix literal (64 floats of input data)

    ex = {}
    stream = torch.cuda.current_stream()
    N = N_SIDE

    def entry(ms, n_px, bytes_per_px, **kw):
        gbs = bytes_per_px * n_px / (ms * 1e-3) / 1e9
        return dict({"ms": ms, "gpixel_s": n_px / (ms * 1e-3) / 1e9, "gb_s": gbs, "frac_of_measured_hbm": gbs / peak,
                     "algorithmic_bytes_per_px": bytes_per_px}, **kw)

    # u8 in / u8 out (2 B/px): issue-bound kernel, the dtype of configs[4]
    ins8 = [torch.randint(0, 256, (N, N), device=dev, dtype=torch.uint8) for _ in range(6)]
    outs8 = [torch.empty_like(x) for x in ins8]
    for key, plan, what in (
            ("u8_8192", m.Plan(), "library default: bit-exact coefficients, factored inverse (u8 pixels within 1 LSB)"),
            ("u8_exact_8192", m.Plan(inverse=m.api.INVERSE_EXACT), "INVERSE_EXACT: u8 pixels bit-identical to the reference"),
            ("u8_k10_8192", m.Plan(keep=m.zigzag_mask(10)), "first 10 zig-zag coefficients retained (compile-time mask kernel)")):
        ms = time_config(m, rotating(m, plan, ins8, outs8, stream))
        ex[key] = entry(ms, N * N, 2, what=what, kernel_path=m.api.last_path())
    del ins8, outs8
    # colour: interleaved RGB u8 -> YCbCr -> three planes (luma / chroma tables) -> RGB, one pass (6 B/px)
    rgb_in = [torch.randint(0, 256, (N, N, 3), device=dev, dtype=torch.uint8) for _ in range(2)]
    rgb_out = [torch.empty_like(x) for x in rgb_in]
    plan_rgb = m.Plan()

    def rgb_step(i):
        m.roundtrip_rgb(rgb_in[i % 2], out=rgb_out[i % 2], plan=plan_rgb, stream=stream)
    ex["rgb_8192"] = entry(time_config(m, rgb_step), N * N, 6, what="b200dct_roundtrip_rgb: 8192^2 RGB pixels (3 planes) per pass, library default inverse",
                           kernel_path=m.api.last_path())
    del rgb_in, rgb_out
    # the drop-in two-call API (dct_all_blocks_cuda then idct_all_blocks_cuda), f32, 16 B/px
    a = [torch.randint(0, 256, (N, N), device=dev, dtype=torch.int32).float() for _ in range(2)]
    c = [torch.empty(N, N, device=dev) for _ in range(2)]
    b = [torch.empty(N, N, device=dev) for _ in range(2)]
    plan = m.Plan()

    def split(i):
        m.forward(a[i % 2], coef=c[i % 2], plan=plan, stream=stream)
        m.inverse(c[i % 2], img=b[i % 2], plan=plan, stream=stream)
    ex["split_forward_inverse_f32_8192"] = entry(time_config(m, split), N * N, 16, what="b200dct_forward + b200dct_inverse, f32 coefficient plane in between")
    # exact DCT (dense DCT-II matrix as data), CUDA cores: configs[3]
    T = o.dct2_T()
    for key, plan, what in (("dense_dct2_8192", m.Plan(T=T), "dense DCT-II, even/odd (symmetric) kernels"),
                            ("dense_dct2_chain_8192", m.Plan(T=T, dense=m.api.DENSE_CHAIN), "dense DCT-II, ordered FMA chains")):
        ms = time_config(m, rotating(m, plan, a, b, stream))
        ex[key] = entry(ms, N * N, 8, what=what, kernel_path=m.api.last_path())
    del a, b, c
    torch.cuda.empty_cache()
    N2 = 16384
    a = [torch.randint(0, 256, (N2, N2), device=dev, dtype=torch.int32).float()]
    b = [torch.empty(N2, N2, device=dev)]
    for key, plan, what in (("dense_dct2_16384", m.Plan(T=T), "BASELINE configs[3]: exact DCT on 16384^2 f32, even/odd (symmetric) CUDA-core kernels"),
                            ("dense_dct2_chain_16384", m.Plan(T=T, dense=m.api.DENSE_CHAIN), "same, ordered FMA chains"),
                            ("sparse_16384", m.Plan(), "HpApprDCT on the same image: identical I/O, strictly less math (lower bound for any dense kernel)")):
        ms = time_config(m, rotating(m, plan, a, b, stream), k=10)
        ex[key] = entry(ms, N2 * N2, 8, what=what, kernel_path=m.api.last_path())
    del a, b
    torch.cuda.empty_cache()
    # SURVEY 8(f2): MSE / PEEN / non-zero count from the same pass (one launch on either family), and 8(f4): images
    # whose sides are not multiples of 8 and whose rows are not aligned (one pass of the edge-replicating kernels)
    import ctypes as C
    L = m.lib()
    for key, dt, code, es, bpp in (("metrics_f32_8192", torch.float32, 0, 4, 8), ("metrics_u8_8192", torch.uint8, 1, 1, 2)):
        xs = [torch.randint(0, 256, (N, N), device=dev, dtype=torch.int32).to(dt) for _ in range(3)]
        ys = [torch.empty_like(x) for x in xs]
        nb = int(L.b200dct_metrics_workspace_bytes(N, N))
        ws = torch.empty(max(1, nb // 8), dtype=torch.float64, device=dev)
        acc = torch.zeros(3, dtype=torch.float64, device=dev)
        sp, plan_m = C.c_void_p(stream.cuda_stream), m.Plan()

        def mstep(i):
            m.api._check(L.b200dct_roundtrip_metrics(plan_m._h, xs[i % 3].data_ptr(), code, N * es, ys[i % 3].data_ptr(), code, N * es,
                                                     None, 0, 0, N, N, acc.data_ptr(), ws.data_ptr(), nb, sp))
        ms = time_config(m, mstep)
        ex[key] = entry(ms, N * N, bpp, launches=m.api.last_launch_count(), kernel_path=m.api.last_path(),
                        what="b200dct_roundtrip_metrics: fused round trip that also accumulates sum (x-y)^2, sum x^2 and the non-zero coefficient count")
        del xs, ys, ws
    M1 = N - 1
    for key, dt, bpp in (("any_f32_8191", torch.float32, 8), ("any_u8_8191", torch.uint8, 2)):
        xs = [torch.randint(0, 256, (M1, M1), device=dev, dtype=torch.int32).to(dt) for _ in range(3)]
        ys = [torch.empty_like(x) for x in xs]
        plan_a = m.Plan()

        def astep(i):
            m.roundtrip_any(xs[i % 3], out=ys[i % 3], plan=plan_a, stream=stream)
        ex[key] = entry(time_config(m, astep), M1 * M1, bpp, kernel_path=m.api.last_path(),
                        what="b200dct_roundtrip_any on an 8191 x 8191 image (sides not multiples of 8, rows unaligned): edge replication, one pass, no scratch image")
        del xs, ys
    torch.cuda.empty_cache()
    # batches of SEPARATELY ALLOCATED images in one launch per 64 images (b200dct_roundtrip_batch) against
    # the loop of single-image calls a caller of the reference writes; the 64 x 8192^2 u8 batch is the
    # alternative form of BASELINE configs[4] on one GPU
    plan = m.Plan()
    for key, n, side, dt, bpp, k in (("batch64_f32_1024", 64, 1024, torch.float32, 8, 20), ("batch64_u8_2048", 64, 2048, torch.uint8, 2, 20),
                                     ("batch64_u8_8192", 64, 8192, torch.uint8, 2, 5)):
        imgs = [torch.randint(0, 256, (side, side), device=dev, dtype=torch.int32).to(dt) for _ in range(n)]
        batch = m.ImageBatch(imgs)

        def bstep(i):
            batch.run(plan=plan, stream=stream)

        def lstep(i):
            for x, y in zip(batch.imgs, batch.outs):
                m.roundtrip(x, out=y, plan=plan, stream=stream)
        ms = time_config(m, bstep, k=k)
        launches = m.api.last_launch_count()
        ex[key] = entry(ms, n * side * side, bpp, launches=launches, kernel_path=m.api.last_path(),
                        loop_of_single_calls_ms=time_config(m, lstep, k=max(2, k // 4), warm=1),
                        what=f"{n} separately allocated {side}^2 {'f32' if dt == torch.float32 else 'u8'} images, one batch call "
                             f"({launches} launch) vs a Python loop of {n} b200dct_roundtrip calls")
        del imgs, batch
        torch.cuda.empty_cache()
    return ex


def extras_multi_gpu(m, dev, rank, world):
    """BASELINE configs[4]: ONE 32768 x 32768 uint8 image striped by block-rows over the ranks
    (strong scaling), every rank's stripe checked against the oracle; plus the optional gather
    fused into the transform (peer stores into rank 0's image over NVLink), once, with parity."""
    import numpy as np
    import torch

    from oracle import oracle as o

    H = Wd = 32768
    r0, r1 = m.stripe_rows(H, world, rank)
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    img = torch.randint(0, 256, (r1 - r0, Wd), device=dev, generator=g, dtype=torch.uint8)
    out = torch.empty_like(img)
    plan = m.Plan()
    stream = torch.cuda.current_stream()

    def step(i):
        m.roundtrip(img, out=out, plan=plan, stream=stream)

    step(0)
    m.dist.barrier()
    torch.cuda.synchronize()
    ms = statistics.median(timed_windows(step, [10] * 3, stream, warm=3)) / 10
    m.dist.barrier()
    ms = m.dist.max_over_ranks(ms, dev)

    def band_ok(t, a):          # u8 pixels within 1 LSB of the oracle (library default: factored inverse)
        want = o.roundtrip(img[a:a + 16].cpu().numpy())
        got = t[a:a + 16].cpu().numpy()
        return int(np.abs(got.astype(np.int16) - want.astype(np.int16)).max()) <= 1

    ok = band_ok(out, 0) and band_ok(out, (r1 - r0) - 16)
    ex = {"u8_32768_strong": {"ms": ms, "gpixel_s": H * Wd / (ms * 1e-3) / 1e9, "rows_per_gpu": r1 - r0,
                              "what": f"one {H}x{Wd} u8 image striped over {world} GPUs, fused round trip, no collective; slowest rank",
                              "parity_all_ranks": m.dist.sum_over_ranks(0.0 if ok else 1.0, dev) == 0.0,
                              "parity_criterion": "coefficients bit-exact by construction; u8 pixels within 1 LSB of the oracle (2 bands per rank)"}}
    # the alternative form of configs[4]: a batch of 64 separately allocated 8192^2 u8 images, image b on
    # rank b mod world (SURVEY section 8e), every rank ONE batch call; strong scaling, no collective
    nb, side = 64, 8192
    mine = m.batch_images(nb, world, rank)
    gb = torch.Generator(device=dev).manual_seed(2000 + rank)
    batch = m.ImageBatch([torch.randint(0, 256, (side, side), device=dev, generator=gb, dtype=torch.uint8) for _ in mine])

    def bstep(i):
        batch.run(plan=plan, stream=stream)

    bstep(0)
    m.dist.barrier()
    torch.cuda.synchronize()
    bms = statistics.median(timed_windows(bstep, [5] * 3, stream, warm=2)) / 5
    m.dist.barrier()
    bms = m.dist.max_over_ranks(bms, dev)
    bok = all(int(np.abs(batch.outs[j][a:a + 16].cpu().numpy().astype(np.int16)
                         - o.roundtrip(batch.imgs[j][a:a + 16].cpu().numpy()).astype(np.int16)).max()) <= 1
              for j in (0, len(mine) - 1) for a in (0, side - 16))
    ex["u8_batch64_8192_strong"] = {"ms": bms, "gpixel_s": nb * side * side / (bms * 1e-3) / 1e9, "images_per_gpu": len(mine),
                                    "launches_per_gpu": m.api.last_launch_count(),
                                    "what": f"{nb} separately allocated {side}^2 u8 images, image b on rank b mod {world}, one b200dct_roundtrip_batch call per rank; slowest rank",
                                    "parity_all_ranks": m.dist.sum_over_ranks(0.0 if bok else 1.0, dev) == 0.0}
    del batch
    torch.cuda.empty_cache()
    try:
        peer = m.dist.PeerImage(H, Wd, torch.uint8, dev)
        dst = peer.stripe_on(0, r0, r1)               # rows [r0, r1) of rank 0's full image

        def fstep(i):
            m.roundtrip(img, out=dst, plan=plan, stream=stream)
            peer.barrier()

        fstep(0)
        torch.cuda.synchronize()
        m.dist.barrier()
        fms = statistics.median(timed_windows(fstep, [5] * 3, stream, warm=1)) / 5
        m.dist.barrier()
        fms = m.dist.max_over_ranks(fms, dev)
        fok = True
        if rank == 0:       # rank 0 holds the assembled image: its own stripe's bands can be checked here
            full = peer.local()
            fok = band_ok(full[r0:r1], 0) and band_ok(full[r0:r1], (r1 - r0) - 16)
        # every other rank checks the bands it wrote by reading them back through the peer mapping
        else:
            fok = band_ok(dst, 0) and band_ok(dst, (r1 - r0) - 16)
        ex["fused_gather_ms"] = fms
        ex["fused_gather_parity"] = m.dist.sum_over_ranks(0.0 if fok else 1.0, dev) == 0.0
        ex["fused_gather_what"] = ("transform whose output plane is a peer-mapped view of rank 0's 1 GiB image "
                                   "(symmetric memory over NVLink/NVSwitch): transform + gather in one kernel, per step, incl. the cross-rank barrier")
    except Exception as e:  # pragma: no cover
        ex["fused_gather_error"] = repr(e)
    return ex


def cpu_baseline():
    from oracle import oracle as o

    o.build()
    img = o.rand_image(N_SIDE, N_SIDE, 42)
    t = o.time_roundtrip(img, reps=3, threads=1)     # ~2 s per pass: ~10 s of CPU work in total
    return {"value": N_SIDE * N_SIDE / t / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "the whole 8192x8192 f32 image (srand(42) rand()%256), best of 3 passes, 1 thread",
            "seconds_per_pass": t, "host_threads_available": len(os.sched_getaffinity(0)),
            "what": "sequential C restatement of the reference's arithmetic (oracle/dct_oracle.c); the reference "
                    "itself has no CPU implementation (SURVEY.md S1)"}


def reference_gpu_kernels(d_img, d_out):
    """The unmodified reference kernels on the same B200: its own printed event times."""
    try:
        import torch

        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import refgpu
        from oracle import oracle as o

        if not refgpu.available("newappr"):
            return None
        refgpu.set_quant("newappr", o.jpeg_Q())
        T = torch.from_numpy(o.haweel_T()).cuda()
        img = d_img.clone()
        coef = torch.empty_like(img)
        res = {}
        for variant in ("newappr", "fastappr"):
            if not refgpu.available(variant):
                continue
            ts = []
            for _ in range(4):
                img.copy_(d_img)
                _, t1 = refgpu.dct(variant, img, T, coef)
                _, t2 = refgpu.idct(variant, coef, T, d_out)
                ts.append(t1 + t2)
            ms = min(ts[1:])
            res[variant] = {"dct_plus_idct_ms": ms, "gpixel_s": N_SIDE * N_SIDE / (ms * 1e-3) / 1e9}
        res["what"] = ("reference kernels compiled unmodified for sm_100a (oracle/_ref), 8192^2 f32 resident in HBM, "
                       "its own cudaEvent times for dct_all_blocks_cuda + idct_all_blocks_cuda (6 launches, 48 B/px)")
        return res
    except Exception as e:  # pragma: no cover
        return {"unavailable": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: 200; 10 for --impl reference, 20 for --impl reference-gpu)")
    ap.add_argument("--warmup", type=int, default=None, help="untimed steps first (default: 10; 3 for --impl reference)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--no-baselines", action="store_true", help="skip the CPU / reference-GPU baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help=f"after the timed steps, write {DUMP_ROWS} fixed rows in all (seeded choice, {DUMP_ROWS}/N per rank) "
                         "of the image the last timed step returned to DIR/out_rank<rank>.npy (float32, 32 MiB in all); "
                         "the inputs are the same in every run")
    args = ap.parse_args()
    steps, warmup = {"ours": (200, 10), "reference": (10, 3), "reference-gpu": (20, 10)}[args.impl]
    args.steps = steps if args.steps is None else args.steps
    args.warmup = warmup if args.warmup is None else args.warmup
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the default arm (--impl ours)")
    if args.impl == "reference":
        return run_reference_cpu(args)
    if args.impl == "reference-gpu":
        return run_reference_gpu(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
