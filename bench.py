#!/usr/bin/env python3
"""bench.py — PageRank GTEPS (edges/sec/iter) on synthetic RMAT, the headline metric of BASELINE.json.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--scale S] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one graph: `page_rank` with 20 forced sweeps
(tolerance 0, damping 0.85) on the RMAT scale-S graph (default 26 = the configuration the metric is
quoted on; it fits one B200).  One JSON line is printed by rank 0.

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (float32, or float64 for
integer results), so that two builds can be compared output for output: the inputs are generated from a
fixed seed.  An output of more than 2**22 entries is cut to a fixed, seeded sample of its entries.

  value        m * sweeps * K / device time of K steps, graph resident in HBM, result left in HBM
  e2e          same metric through the C ABI with HOST buffers (gb_page_rank_csr_u32): every step uploads
               the pinned host in-CSR + out offsets, builds the device layout, runs page_rank and
               copies the ranks back; nothing stays resident between steps
  roofline     the sweep kernels (k_pr_cb + k_pr_sell + k_pr_finish) timed with CUDA events around every sweep:
               algorithmic bytes (4m + 24n + 4 per sweep) / mean launch time vs measured HBM peak
  cpu_baseline the reference's multi-threaded in-place sweep (oracle.page_rank_mt, the C restatement
               of crates/algos/src/page_rank.rs:113-168) on the same graph, bounded sample
  --impl reference   times that CPU path alone, all host threads, same metric / config
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SWEEPS = 20
PR_KERNEL_VERSION = "r02-cb16"   # bump with every change of the sweep kernels / layout (keys profiles/pr_traffic.json)
DAMPING = 0.85
SEED = 42
EDGE_FACTOR = 16


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every 20 ms while the timed region runs
    (nvidia-smi -lms is too slow to land a sample inside a 0.1 s region)."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES-relative index -> NVML handle via the PCI bus id of the torch device
            import torch
            bus = torch.cuda.get_device_properties(self.index).pci_bus_id if hasattr(
                torch.cuda.get_device_properties(self.index), "pci_bus_id") else None
            h = None
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    cand = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if int(pynvml.nvmlDeviceGetPciInfo(cand).bus) == int(bus):
                        h = cand
                        break
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self._nv, self._h = pynvml, h
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None
        return self

    def _loop(self):
        nv, h = self._nv, self._h
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def pinned_empty(count: int, dtype):
    """numpy view of pinned host memory (torch owns the allocation)."""
    import torch
    tdt = {np.uint32: torch.int32, np.float32: torch.float32}[dtype]
    t = torch.empty(max(count, 1), dtype=tdt, pin_memory=torch.cuda.is_available())
    return t, t.numpy().view(dtype)[:count]


DUMP_SAMPLE = 1 << 22       # entries --dump-outputs keeps of one output array
DUMP_BUDGET = 64 << 20      # bytes --dump-outputs may write in all


def dump_index(n: int) -> np.ndarray:
    """Sorted indices of the entries --dump-outputs keeps of an n-entry output: all of them up to
    DUMP_SAMPLE, else a sample drawn from a fixed seed (the same indices on every run)."""
    if n <= DUMP_SAMPLE:
        return np.arange(n)
    return np.unique(np.random.default_rng(SEED).integers(0, n, DUMP_SAMPLE))


def dump_outputs(path, outputs: dict) -> None:
    """Writes every output as path/<name>.npy: float32 stays float32, everything else becomes float64
    (exact for integers below 2**53)."""
    arrays = {}
    for name, a in outputs.items():
        a = np.asarray(a)
        arrays[name] = a if a.dtype == np.float32 else a.astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BUDGET:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_BUDGET} byte budget")
    out = Path(path)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


def algorithmic_bytes(n: int, m: int) -> int:
    return 4 * m + 24 * n + 4  # BASELINE.md §3 / SURVEY.md §8(d)


def cpu_leg(out_off, in_off, in_tgt, n, m, sweeps, threads=0):
    """The reference's multi-threaded in-place sweep on the host cores (bounded sample)."""
    import oracle
    oracle.page_rank_mt(in_off, in_tgt, out_off, 1, 0.0, DAMPING, threads)  # warm-up sweep
    t0 = time.perf_counter()
    _, it, _ = oracle.page_rank_mt(in_off, in_tgt, out_off, sweeps, 0.0, DAMPING, threads)
    dt = time.perf_counter() - t0
    return m * it / dt / 1e9, dt, oracle.hardware_threads() if threads == 0 else threads


def verify_last_sweep(g, d_scores, in_off, in_tgt, out_off, n, samples=4096, rtol=1e-6):
    """Untimed check of the benchmarked result: sweep 20 of sampled rows is re-evaluated in f64 on the
    host from the out_scores of a 19-sweep run (deterministic, so its scores are sweep 20's inputs).
    d_scores holds the 20-sweep ranks of the timed runs."""
    import torch
    from graph_b200 import _capi
    from graph_b200._capi import lib, check
    s20 = d_scores.cpu().numpy()
    it, err = C.c_uint64(0), C.c_double(0.0)
    cfg19 = _capi.PageRankConfig(SWEEPS - 1, 0.0, DAMPING, _capi.PR_JACOBI)
    d19 = torch.empty(n, dtype=torch.float32, device="cuda")
    check(lib.gb_page_rank_device(g._g, C.byref(cfg19), C.c_void_p(d19.data_ptr()), C.byref(it), C.byref(err)))
    s19 = d19.cpu().numpy()
    outdeg = np.diff(out_off.astype(np.int64)).astype(np.float32)
    with np.errstate(divide="ignore"):
        x19 = s19 / outdeg                       # f32 IEEE division, as the kernel's __fdiv_rn
    indeg = np.diff(in_off.astype(np.int64))
    rng = np.random.default_rng(7)
    rows = np.unique(np.concatenate([rng.integers(0, n, samples), np.argpartition(indeg, -64)[-64:]]))
    base = (np.float32(1.0) - np.float32(DAMPING)) / np.float32(n)
    worst = 0.0
    for u in rows:
        tot = np.float32(x19[in_tgt[in_off[u]:in_off[u + 1]]].astype(np.float64).sum())
        want = np.float32(base + np.float32(np.float32(DAMPING) * tot))
        worst = max(worst, abs(float(s20[u]) - float(want)) / float(want))
    ok = bool(worst <= rtol and np.isfinite(s20).all())
    return ok, {"rows": int(len(rows)), "max_rel_err": worst, "rtol": rtol,
                "what": "sweep 20 of sampled rows (random + the 64 largest hubs) re-evaluated in f64 on the host "
                        "from a 19-sweep run's out_scores"}


def host_csr_from_device(g, pinned=True, out_targets=True):
    """(out_off, out_tgt, in_off, in_tgt) host copies of a DiGraph's CSR pair, pinned when possible
    (out_tgt is None when out_targets is False: page_rank reads only the out-degrees)."""
    from graph_b200._capi import lib, check, CSR_OUT, CSR_IN
    n, m = g.node_count(), g.edge_count()
    keep, arrs = [], []
    for which in (CSR_OUT, CSR_IN):
        t_off, off = pinned_empty(n + 1, np.uint32)
        want_tgt = out_targets or which == CSR_IN
        t_tgt, tgt = pinned_empty(m, np.uint32) if want_tgt else (None, None)
        check(lib.gb_graph_copy_csr(g._g, which, off.ctypes.data_as(C.c_void_p),
                                    tgt.ctypes.data_as(C.c_void_p) if want_tgt else None, None))
        keep += [t_off, t_tgt]
        arrs += [off, tgt]
    return arrs, keep


# ---------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; the Rust crate cannot be built here)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    scale, n = args.scale, 1 << args.scale
    m = EDGE_FACTOR * n
    # input preparation (untimed): the device generator/CSR builder when a GPU is present, else the
    # oracle's own single-threaded builder
    try:
        import torch
        import graph_b200 as gb
        if not torch.cuda.is_available():
            raise RuntimeError("no gpu")
        g = gb.DiGraph.rmat(scale, EDGE_FACTOR, SEED, gb.Layout.Sorted)
        (out_off, _out_tgt, in_off, in_tgt), keep = host_csr_from_device(g, pinned=False)
        del g
        prep = "device generator + CSR build (untimed)"
    except Exception:
        src, dst = oracle.rmat_edges(scale, SEED)
        out_off, _ = oracle.csr_build(src, dst, n, oracle.OUTGOING, oracle.SORTED)
        in_off, in_tgt = oracle.csr_build(src, dst, n, oracle.INCOMING, oracle.SORTED)
        prep = "oracle generator + CSR build (untimed)"
    sample_sweeps = args.ref_sweeps
    threads = oracle.hardware_threads()
    for _ in range(args.warmup):
        oracle.page_rank_mt(in_off, in_tgt, out_off, 1, 0.0, DAMPING, 0)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        scores, it, err = oracle.page_rank_mt(in_off, in_tgt, out_off, sample_sweeps, 0.0, DAMPING, 0)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"scores": scores[dump_index(n)], "iterations": [it], "error": [err]})
    gteps = m * sample_sweeps * args.steps / dt / 1e9
    sample = f"{sample_sweeps} of {SWEEPS} sweeps per step on the full RMAT scale-{scale} graph; input prep: {prep}"
    line = {
        "impl": "reference", "metric": "PageRank GTEPS (edges/sec/iter)", "value": gteps, "unit": "GTEPS",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(scale, 0),
        "cpu_baseline": {"value": gteps, "unit": "GTEPS", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": gteps, "unit": "GTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(scale, n_gpus):
    n = 1 << scale
    return {"workload": f"page_rank f32, RMAT scale-{scale} (n={n}, m={EDGE_FACTOR * n}), {SWEEPS} sweeps forced "
                        f"(tolerance 0), damping {DAMPING}, CsrLayout::Sorted, seed {SEED}",
            "scale": scale, "sweeps": SWEEPS, "damping": DAMPING, "schedule": "jacobi",
            "l2": "inputs larger than L2 (target stream >= 256 MiB per sweep), no explicit flush",
            "parallelism": f"edge-cut x{n_gpus}" if n_gpus > 1 else "single GPU"}


# ---------------------------------------------------------------------------------------------
def run_single(args):
    import torch
    import graph_b200 as gb
    from graph_b200 import _capi
    from graph_b200._capi import lib, check
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(0)
    gb.set_device(0)
    scale, n = args.scale, 1 << args.scale
    m = EDGE_FACTOR * n
    g = gb.DiGraph.rmat(scale, EDGE_FACTOR, SEED, gb.Layout.Sorted)
    cfg = _capi.PageRankConfig(SWEEPS, 0.0, DAMPING, _capi.PR_JACOBI)
    d_scores = torch.empty(n, dtype=torch.float32, device="cuda")
    it, err = C.c_uint64(0), C.c_double(0.0)
    stream = torch.cuda.ExternalStream(g.cuda_stream())

    def step():
        check(lib.gb_page_rank_device(g._g, C.byref(cfg), C.c_void_p(d_scores.data_ptr()), C.byref(it), C.byref(err)))
        return g.last_timing()

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    with ClockSampler(0) as clocks:
        torch.cuda.synchronize()
        ev0.record(stream)
        for _ in range(args.steps):
            launches += step()["kernel_launches"]
        ev1.record(stream)
        torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    assert it.value == SWEEPS
    gteps = m * SWEEPS * args.steps / (ms * 1e-3) / 1e9
    if args.dump_outputs:   # taken before the passes below run the step again
        idx = torch.from_numpy(dump_index(n)).to(d_scores.device)
        outputs = {"scores": d_scores[idx].cpu().numpy(), "iterations": [it.value], "error": [err.value]}

    # dominant kernel, timed live with CUDA events around every launch (separate pass)
    lib.gb_set_profiling(1)
    hot_ms, hot_n = 0.0, 0
    for _ in range(min(args.steps, 3)):
        t = step()
        hot_ms += t["hot_kernel_ms"]
        hot_n += t["hot_kernel_launches"]
    lib.gb_set_profiling(0)
    peak, peak_src = peaks()
    bytes_per_launch = algorithmic_bytes(n, m)
    achieved = bytes_per_launch / (hot_ms / hot_n * 1e-3) / 1e9 if hot_n else 0.0
    # DRAM bytes per sweep from the committed ncu capture of THIS kernel version and layout (else null)
    traffic, traffic_src = None, None
    tp = ROOT / "profiles" / "pr_traffic.json"
    if tp.exists():
        try:
            rec = json.loads(tp.read_text())
            if rec.get("kernel_version") == PR_KERNEL_VERSION:
                traffic = rec.get(f"scale{scale}")
                traffic_src = rec.get("source")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "k_pr_cb + k_pr_sell + k_pr_finish (one sweep)", "achieved": achieved,
                "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_per_launch, "mean_launch_ms": hot_ms / max(hot_n, 1),
                "kernel_share_of_step": (hot_ms / max(min(args.steps, 3), 1)) / (ms / args.steps)}

    layout = g.page_rank_plan_info()
    # e2e through the C ABI with host buffers (pinned): upload + device twin + page_rank + ranks back
    (out_off, out_tgt, in_off, in_tgt), keep = host_csr_from_device(g)
    verified, verification = verify_last_sweep(g, d_scores, in_off, in_tgt, out_off, n)
    del g
    torch.cuda.empty_cache()
    _, h_scores = pinned_empty(n, np.float32)
    cfg_h = _capi.PageRankConfig(SWEEPS, 0.0, DAMPING, _capi.PR_JACOBI)

    def e2e_step():
        check(lib.gb_page_rank_csr_u32(0, n, in_off.ctypes.data_as(C.c_void_p), in_tgt.ctypes.data_as(C.c_void_p),
                                       out_off.ctypes.data_as(C.c_void_p), C.byref(cfg_h),
                                       h_scores.ctypes.data_as(C.c_void_p), C.byref(it), C.byref(err)))

    e2e_steps = max(3, min(args.steps, 5))
    e2e_step()  # warm-up
    torch.cuda.synchronize()
    step_s = []
    for _ in range(e2e_steps):
        t0 = time.perf_counter()
        e2e_step()  # returns after the ranks are back in host memory (the call synchronises)
        step_s.append(time.perf_counter() - t0)
    e2e_med = float(np.median(step_s))  # median step: one PCIe / host hiccup must not decide the figure
    e2e = {"value": m * SWEEPS / e2e_med / 1e9, "unit": "GTEPS",
           "h2d_bytes_per_step": int(4 * m + 8 * (n + 1)), "d2h_bytes_per_step": int(4 * n),
           "steps": e2e_steps, "ms_per_step": e2e_med * 1e3, "ms_per_step_all": [round(t * 1e3, 1) for t in step_s],
           "what": "gb_page_rank_csr_u32: pinned host in-CSR + out offsets -> device, layout build, 20 sweeps, "
                   "ranks back to the host, everything freed (no resident state between steps); median step"}

    # CPU baseline on the same graph, bounded sample
    cpu = None
    if not args.no_cpu:
        v, dt, cores = cpu_leg(out_off, in_off, in_tgt, n, m, args.cpu_sweeps)
        cpu = {"value": v, "unit": "GTEPS", "cores": cores, "kind": "port",
               "sample": f"{args.cpu_sweeps} in-place sweeps (after 1 warm-up sweep) of oracle.page_rank_mt on the "
                         f"same RMAT scale-{scale} CSR, {dt:.2f} s"}

    line = {
        "metric": "PageRank GTEPS (edges/sec/iter)", "value": gteps, "unit": "GTEPS", "n_gpus": 1,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {**workload_config(scale, 1), "layout": layout}, "clocks": clocks.summary(), "e2e": e2e,
        "gpu_launches": int(launches), "verified": verified, "verification": verification,
        "roofline": roofline, "cpu_baseline": cpu,
        "hbm_roofline_gteps": peak * 1e9 / (bytes_per_launch / m) / 1e9,
        "frac_of_hbm_roofline_whole_step": (bytes_per_launch * SWEEPS * args.steps / (ms * 1e-3) / 1e9) / peak,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
def run_multi(args):
    """N > 1: one process per GPU (torchrun), 1-D edge-cut (32-row slices dealt round-robin), fused exchange."""
    import torch
    import torch.distributed as dist
    import graph_b200 as gb
    from graph_b200.multigpu import ShardedPageRank
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    # NCCL prints its version banner on stdout: keep stdout for the ONE JSON line
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    gb.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    scale, n = args.scale, 1 << args.scale
    m = EDGE_FACTOR * n
    g = gb.DiGraph.rmat(scale, EDGE_FACTOR, SEED, gb.Layout.Sorted)
    spr = ShardedPageRank(g, exchange=args.exchange, multicast=not args.no_multicast)
    for _ in range(max(args.warmup, 3)):
        spr.run(SWEEPS, DAMPING)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        dist.barrier()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.steps):
            spr.run(SWEEPS, DAMPING)
        ev1.record()
        torch.cuda.synchronize()
        dist.barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device="cuda", dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    gteps = m * SWEEPS * args.steps / (ms * 1e-3) / 1e9
    stats = spr.backend.stats
    # untimed verification: the sharded ranks against a single-GPU run of the same graph on rank 0
    sharded = spr.scores_host()
    verified, verification = None, None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"scores": sharded[dump_index(n)], "iterations": [spr.ran_iterations],
                                         "error": [spr.error]})
    if rank == 0:
        single = g.page_rank(max_iterations=SWEEPS, tolerance=0.0, damping_factor=DAMPING, mode="jacobi").scores()
        worst = float(np.max(np.abs(sharded - single) / single))
        verified = bool(worst <= 1e-6 and np.isfinite(sharded).all())
        verification = {"max_rel_err_vs_single_gpu": worst, "rtol": 1e-6,
                        "what": f"all {n} ranks of the {world}-GPU run against a 1-GPU run of the same graph on rank 0 "
                                "(itself checked against the oracle at this size by tests/test_gpu_parity.py)"}
    if args.diag:
        spr.diag = []
        spr.run(SWEEPS, DAMPING)
        k_ms, x_ms = spr.diag_summary()
        info = torch.tensor([k_ms, x_ms, float(stats["local_rows"]), float(stats["local_edges"])], device="cuda",
                            dtype=torch.float64)
        allinfo = [torch.zeros_like(info) for _ in range(world)]
        dist.all_gather(allinfo, info)
        if rank == 0:
            print("diag per rank (kernel ms, exchange+wait ms, rows, edges):",
                  [[round(float(v), 3) for v in t] for t in allinfo], file=sys.stderr)
        spr.diag = None
    # e2e, same meaning as at N = 1: nothing is resident between steps.  Every rank holds the page_rank
    # inputs (in-CSR + out offsets) in pinned host memory; a step uploads them, builds this rank's shard
    # layout, runs the sweeps and brings the full score vector back to the host.
    (out_off, _none, in_off, in_tgt), keep = host_csr_from_device(g, out_targets=False)
    del g
    torch.cuda.empty_cache()
    e2e_steps = max(3, min(args.steps, 5))
    step_s = []
    for i in range(e2e_steps + 1):   # the first step is a warm-up
        dist.barrier()
        t0 = time.perf_counter()
        gh = gb.DiGraph.for_page_rank(in_off, in_tgt, out_off)
        spr.rebind(gh)
        spr.run(SWEEPS, DAMPING)
        host = spr.scores_host(reuse=True)   # page-locked, like the N = 1 path's result buffer
        del gh
        dt = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        if i:
            step_s.append(float(dt.item()))
    e2e_med = float(np.median(step_s))
    if rank == 0:
        peak, peak_src = peaks()
        ab = algorithmic_bytes(n, m)
        line = {
            "metric": "PageRank GTEPS (edges/sec/iter)", "value": gteps, "unit": "GTEPS", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {**workload_config(scale, world), "exchange": spr.exchange,
                                            "multicast": spr.multicast, "deal": "32-row slices round-robin",
                                            "layout_rank0": stats},
            "clocks": clocks.summary(),
            "e2e": {"value": m * SWEEPS / e2e_med / 1e9, "unit": "GTEPS",
                    "h2d_bytes_per_step": int(4 * m + 8 * (n + 1)) * world, "d2h_bytes_per_step": int(4 * n) * world,
                    "steps": e2e_steps, "ms_per_step": e2e_med * 1e3,
                    "ms_per_step_all": [round(t * 1e3, 1) for t in step_s],
                    "what": "per step and per rank: pinned host in-CSR + out offsets -> device, this rank's shard "
                            "layout, 20 sweeps with the fused exchange, all ranks' scores summed and copied to the "
                            "host; nothing resident between steps (every rank uploads the whole in-CSR: the storage "
                            "is not sharded on the host side); median step, max over ranks"},
            "gpu_launches": int(spr.launches), "verified": verified, "verification": verification,
            "roofline": {"bound": "hbm", "kernel": "k_pr_cb + k_pr_sell + k_pr_finish + k_pr_sync (one sweep, per rank)",
                         "achieved": ab * SWEEPS * args.steps / (ms * 1e-3) / 1e9,
                         "peak": peak * world, "unit": "GB/s", "frac": ab * SWEEPS * args.steps / (ms * 1e-3) / 1e9 / (peak * world),
                         "traffic": None, "peak_source": peak_src + f" x {world} GPUs, whole step incl. exchange"},
            "cpu_baseline": None,
        }
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    dist.destroy_process_group()


def run_algo(args):
    """--algo wcc | tc | sssp: the other three configs of BASELINE.json on one GPU, one JSON line each, in
    the same shape as the PageRank line (value = device-timed with the graph resident, e2e = through the
    host-buffer call, roofline against BASELINE.md's algorithmic bytes, cpu_baseline = the oracle port)."""
    import torch
    import graph_b200 as gb
    import oracle
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(0)
    gb.set_device(0)
    peak, peak_src = peaks()
    reps = args.steps

    def timed(fn):
        for _ in range(max(args.warmup, 1)):
            fn()
        dev, wall, launches = [], [], 0
        res = None
        for _ in range(reps):
            t0 = time.perf_counter()
            res = fn()
            wall.append(time.perf_counter() - t0)
            t = g.last_timing()
            dev.append(t["total_ms"])
            launches += t["kernel_launches"]
        return res, float(np.median(dev)), float(np.median(wall)) * 1e3, launches

    if args.algo == "wcc":
        scale = args.scale if args.scale != 26 else 24
        n, m = 1 << scale, EDGE_FACTOR << scale
        g = gb.DiGraph.rmat(scale, EDGE_FACTOR, SEED, gb.Layout.Sorted)
        with ClockSampler(0) as clocks:
            res, dev_ms, wall_ms, launches = timed(lambda: g.wcc())
        byts = 8 * m + 16 * n + 8
        comp = res.components()
        outputs = {"components": comp[dump_index(n)]}
        oo, ot = g.csr("out")
        io, it = g.csr("in")
        cpu = None
        verified = None
        if not args.no_cpu:
            oracle.wcc_afforest(oo, ot, io, it, threads=0)
            t0 = time.perf_counter()
            c = oracle.wcc_afforest(oo, ot, io, it, threads=0)
            dt = time.perf_counter() - t0
            verified = bool((c == comp).all())
            cpu = {"value": m / dt / 1e9, "unit": "G edges/s", "cores": oracle.hardware_threads(), "kind": "port",
                   "sample": f"one wcc_afforest run (after one warm-up) on the same CSR pair, {dt:.2f} s"}
        line = {"metric": "WCC (Afforest) G edges/s", "value": m / (dev_ms * 1e-3) / 1e9, "unit": "G edges/s",
                "ms_per_step": dev_ms, "components": int(len(np.unique(comp))),
                "config": {"workload": f"wcc_afforest, directed RMAT scale-{scale} (n={n}, m={m}), defaults 16384/2/1024"},
                "e2e": {"value": m / (wall_ms * 1e-3) / 1e9, "unit": "G edges/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 4 * n, "ms_per_step": wall_ms,
                        "what": "gb_wcc on the resident twin, component ids copied to the host"},
                "roofline": {"bound": "hbm", "kernel": "k_cc_* (whole run)", "achieved": byts / (dev_ms * 1e-3) / 1e9,
                             "peak": peak, "unit": "GB/s", "frac": byts / (dev_ms * 1e-3) / 1e9 / peak, "traffic": None,
                             "peak_source": peak_src, "algorithmic_bytes_per_launch": byts,
                             "note": "Afforest skips most edge lists, so the effective figure can exceed 1"}}
    elif args.algo == "tc":
        scale = args.scale if args.scale != 26 else 22
        n, m = 1 << scale, EDGE_FACTOR << scale
        g = gb.Graph.rmat(scale, EDGE_FACTOR, SEED, gb.Layout.Sorted)
        with ClockSampler(0) as clocks:
            raw, raw_ms, _, l0 = timed(lambda: g.global_triangle_count())
            t0 = time.perf_counter()
            g.make_degree_ordered()
            relabel_ms = (time.perf_counter() - t0) * 1e3
            res, dev_ms, wall_ms, launches = timed(lambda: g.global_triangle_count())
        launches += l0
        outputs = {"triangles": [res.triangles]}
        byts = 8 * m + 4 * (n + 1)
        cpu, verified = None, None
        if not args.no_cpu:
            off, tgt = g.csr()
            t0 = time.perf_counter()
            c = oracle.triangle_count(off, tgt, threads=0)
            dt = time.perf_counter() - t0
            verified = bool(c == res.triangles)
            cpu = {"value": m / dt / 1e9, "unit": "G edges/s", "cores": oracle.hardware_threads(), "kind": "port",
                   "sample": f"one global_triangle_count on the same degree-ordered CSR, {dt:.2f} s"}
        line = {"metric": "triangle count G edges/s (degree-ordered)", "value": m / (dev_ms * 1e-3) / 1e9,
                "unit": "G edges/s", "ms_per_step": dev_ms, "triangles": int(res.triangles),
                "triangles_sorted_layout": int(raw.triangles), "ms_sorted_layout": raw_ms, "relabel_ms": relabel_ms,
                "config": {"workload": f"global_triangle_count, undirected RMAT scale-{scale} (n={n}, 2m={2 * m} entries), "
                                       "CsrLayout::Sorted, after make_degree_ordered"},
                "e2e": {"value": m / (wall_ms * 1e-3) / 1e9, "unit": "G edges/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 8, "ms_per_step": wall_ms, "what": "gb_triangle_count on the resident twin"},
                "roofline": {"bound": "hbm", "kernel": "k_tc", "achieved": byts / (dev_ms * 1e-3) / 1e9, "peak": peak,
                             "unit": "GB/s", "frac": byts / (dev_ms * 1e-3) / 1e9 / peak, "traffic": None,
                             "peak_source": peak_src, "algorithmic_bytes_per_launch": byts,
                             "note": "compulsory bytes only; the kernel is bound by dependent L2 lookups"}}
    else:
        scale = args.scale if args.scale != 26 else 22
        n, m = 1 << scale, EDGE_FACTOR << scale
        g = gb.DiGraph.rmat(scale, EDGE_FACTOR, SEED, gb.Layout.Sorted, weights=True)
        off, _ = g.csr("out")
        start = int(np.argmax(np.diff(off.astype(np.int64))))
        delta = 0.05
        with ClockSampler(0) as clocks:
            res, dev_ms, wall_ms, launches = timed(lambda: g.delta_stepping(start_node=start, delta=delta))
        d = res.distances()
        outputs = {"distances": d[dump_index(n)]}
        byts = 8 * m + 4 * (n + 1) + 8 * n
        cpu, verified = None, None
        if not args.no_cpu:
            off, tgt = g.csr("out")
            w = g.out_weights()
            t0 = time.perf_counter()
            c = oracle.sssp_delta_stepping(off, tgt, w, start, delta)
            dt = time.perf_counter() - t0
            verified = bool(c.tobytes() == d.tobytes())
            cpu = {"value": m / dt / 1e9, "unit": "G edges/s", "cores": 1, "kind": "port",
                   "sample": f"one delta_stepping run (single thread) on the same weighted CSR, {dt:.2f} s"}
        line = {"metric": "delta-stepping SSSP G edges/s", "value": m / (dev_ms * 1e-3) / 1e9, "unit": "G edges/s",
                "ms_per_step": dev_ms, "reached": int((d < np.finfo(np.float32).max).sum()),
                "config": {"workload": f"delta_stepping, weighted RMAT scale-{scale} (n={n}, m={m}), delta {delta}, "
                                       "start = max out-degree vertex"},
                "e2e": {"value": m / (wall_ms * 1e-3) / 1e9, "unit": "G edges/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 4 * n, "ms_per_step": wall_ms,
                        "what": "gb_sssp on the resident twin, distances copied to the host"},
                "roofline": {"bound": "hbm", "kernel": "k_sssp_* (whole run)", "achieved": byts / (dev_ms * 1e-3) / 1e9,
                             "peak": peak, "unit": "GB/s", "frac": byts / (dev_ms * 1e-3) / 1e9 / peak, "traffic": None,
                             "peak_source": peak_src, "algorithmic_bytes_per_launch": byts,
                             "note": "frontier driven: one launch per pass of a bucket"}}
    line.update({"algo": args.algo, "n_gpus": 1, "steps": reps, "warmup": max(args.warmup, 1), "higher_is_better": True,
                 "scaling": "strong", "vs_baseline": None, "dtype": "u32" if args.algo != "sssp" else "f32",
                 "data": "synthetic", "clocks": clocks.summary(), "gpu_launches": int(launches),
                 "verified": verified, "cpu_baseline": cpu})
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scale", type=int, default=26)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--algo", default="page_rank", choices=["page_rank", "wcc", "tc", "sssp"],
                    help="page_rank = the headline line; wcc / tc / sssp = the other BASELINE.json configs (1 GPU)")
    ap.add_argument("--cpu-sweeps", type=int, default=3, help="sweeps of the CPU baseline sample")
    ap.add_argument("--ref-sweeps", type=int, default=5, help="sweeps per step of --impl reference")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "allgather"])
    ap.add_argument("--no-multicast", action="store_true", help="multi-GPU: unicast peer stores instead of multimem.st")
    ap.add_argument("--diag", action="store_true", help="multi-GPU: print per-rank kernel / exchange ms per sweep")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (larger outputs: a seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    elif args.algo != "page_rank":
        run_algo(args)
    elif args.gpus > 1 or int(os.environ.get("WORLD_SIZE", "1")) > 1:
        run_multi(args)
    else:
        run_single(args)


if __name__ == "__main__":
    main()
