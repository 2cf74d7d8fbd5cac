"""pr_knobs.py — time the JACOBI sweep under several layout knobs on one resident graph.

  python tools/pr_knobs.py --scale 26 --configs "B=32768,TAU=3;B=32768,TAU=2;B=49152,TAU=3"

Prints one JSON line per configuration: layout statistics, ms per sweep (CUDA events around every
sweep: k_pr_cb + k_pr_sell + k_pr_finish), GTEPS and the fraction of the HBM roofline."""
import argparse
import ctypes as C
import json
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=int, default=26)
    ap.add_argument("--configs", default="B=32768,TAU=3")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    import graph_b200 as gb
    from graph_b200 import _capi
    from graph_b200._capi import lib, check
    n = 1 << args.scale
    m = 16 * n
    g = gb.DiGraph.rmat(args.scale, 16, 42, gb.Layout.Sorted)
    d_scores = torch.empty(n, dtype=torch.float32, device="cuda")
    cfg = _capi.PageRankConfig(20, 0.0, 0.85, _capi.PR_JACOBI)
    it, err = C.c_uint64(0), C.c_double(0.0)
    peak = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())["hbm_gbs"] if (ROOT / "MEASURED_PEAKS.json").exists() else 6650.0
    names = {"B": "GB_PR_BLOCK", "TAU": "GB_PR_TAU", "CHUNK": "GB_PR_CHUNK"}
    for conf in args.configs.split(";"):
        for k in names.values():
            os.environ.pop(k, None)
        for kv in filter(None, conf.split(",")):
            k, v = kv.split("=")
            os.environ[names[k]] = v
        check(lib.gb_page_rank_plan_reset(g._g))
        info = g.page_rank_plan_info()
        lib.gb_set_profiling(0)
        check(lib.gb_page_rank_device(g._g, C.byref(cfg), C.c_void_p(d_scores.data_ptr()), C.byref(it), C.byref(err)))
        lib.gb_set_profiling(1)
        best, tot = 1e30, []
        for _ in range(args.reps):
            check(lib.gb_page_rank_device(g._g, C.byref(cfg), C.c_void_p(d_scores.data_ptr()), C.byref(it), C.byref(err)))
            t = g.last_timing()
            ms = t["hot_kernel_ms"] / max(t["hot_kernel_launches"], 1)
            best = min(best, ms)
            tot.append(round(t["total_ms"], 3))
        lib.gb_set_profiling(0)
        bytes_alg = 4 * m + 24 * n + 4
        print(json.dumps({"config": conf, "scale": args.scale, "ms_per_sweep": round(best, 4),
                          "gteps": round(m / (best * 1e-3) / 1e9, 1),
                          "roofline_frac": round(bytes_alg / (best * 1e-3) / 1e9 / peak, 4),
                          "total_ms_20_sweeps": tot, "err": err.value, "layout": info}), flush=True)


if __name__ == "__main__":
    main()
