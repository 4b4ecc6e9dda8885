"""K7 (one thread-block cluster per LP) against today's per-LP path, on batches of mid-size LPs.

(a) one ``solve_batched(tables, n, m, engine="cluster")`` call for the whole batch;
(b) one ``SimplexMethod(rows, c, engine="stream").solve()`` per LP (auto loop: the L2-resident
    kernel K5 at these sizes).
Both are warmed up, then run alternately --reps times in this process; times are host clocks that end
in a device synchronise and include uploads and result downloads.  Every LP's status, trace, final
table bits and x from (a) must equal (b)'s, and every forced cluster size that fits must give (a)'s bits.
Prints one JSON line per workload.

    python tools/cluster_bench.py [--reps 3] [--max-lps N] [--workloads p1_100x100,d_128x256,...]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from simplex_method_solver_b200 import workloads as W  # noqa: E402

# name -> (LPs, generator, n, m, max_pivots); the phase-1 family at 100 x 100 is just over K4's 10,000 cells
WORKLOADS = {
    "p1_100x100": (1024, W.phase1_lp, 100, 100, 2000),
    "d_128x256": (256, W.dense_lp, 128, 256, 4000),
    "d_256x512": (64, W.dense_lp, 256, 512, 10000),
    "d_400x800": (16, W.dense_lp, 400, 800, 20000),
}
OPT_CLUSTER_SIZE = 16


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def footprint_sizes(L, n, m):
    """Every cluster size whose footprint fits (include/spx_b200.h)."""
    out = []
    for S in (1, 2, 4, 8, 16):
        assert L.spx_set_option(OPT_CLUSTER_SIZE, S) == 0
        try:
            # validation only: B = 0 launches nothing
            if L.spx_solve_batched_cluster(None, 0, n, m, 0, 0, None, None, None, None, None, None, None, None,
                                           None) == 0:
                out.append(S)
        finally:
            L.spx_set_option(OPT_CLUSTER_SIZE, 0)
    return out


def run_a(tables, n, m, cap):
    import torch
    from simplex_method_solver_b200.batched import solve_batched
    t0 = time.perf_counter()
    res = solve_batched(tables, n, m, max_pivots=cap, engine="cluster")
    torch.cuda.synchronize()
    return time.perf_counter() - t0, res


def run_b(lps, cap):
    import torch
    from simplex_method_solver_b200.simplex import SimplexMethod
    out = []
    t0 = time.perf_counter()
    for rows, c in lps:
        sm = SimplexMethod(rows, c, engine="stream")
        sol = sm.solve(max_pivots=cap)
        out.append((sol, sm))
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def check_equal(res, outs, n, m):
    for k, (sol, sm) in enumerate(outs):
        assert int(res.status[k]) == sol.status and int(res.npiv[k]) == sol.npiv, k
        assert res.trace[k, : sol.npiv].tobytes() == np.ascontiguousarray(sol.trace, dtype=np.int32).tobytes(), k
        flat = np.concatenate([np.asarray(r, dtype=np.float64) for r in sm.table])
        assert res.tables[k].tobytes() == flat.tobytes(), k
        assert res.x[k].tobytes() == np.asarray(sol.x, dtype=np.float64).tobytes(), k


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--max-lps", type=int, default=0, help="cap the LPs of every workload (0: as listed)")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    import torch
    from simplex_method_solver_b200 import _native as N
    L = N.lib()
    gpu = gpu_info()
    for name in args.workloads.split(","):
        B, gen, n, m, cap = WORKLOADS[name]
        if args.max_lps:
            B = min(B, args.max_lps)
        lps = [gen(n, m, seed) for seed in range(B)]
        tables = np.stack([np.concatenate([r.reshape(-1), c]) for r, c in lps])
        cells = n * (m + 1) + m
        S = L.spx_cluster_size(n, m)
        # warm-up of both paths
        run_a(tables, n, m, cap)
        run_b(lps[:2], cap)
        ta, tb = [], []
        for _ in range(args.reps):
            t, res = run_a(tables, n, m, cap)
            ta.append(t)
            t, outs = run_b(lps, cap)
            tb.append(t)
        check_equal(res, outs, n, m)
        # forced cluster sizes: same bits, time of each
        sweep = {}
        for s in footprint_sizes(L, n, m):
            assert L.spx_set_option(OPT_CLUSTER_SIZE, s) == 0
            try:
                run_a(tables, n, m, cap)
                ts = []
                for _ in range(args.reps):
                    t, r2 = run_a(tables, n, m, cap)
                    ts.append(t)
            finally:
                L.spx_set_option(OPT_CLUSTER_SIZE, 0)
            for f in ("status", "npiv", "trace", "tables", "x", "obj", "rowlab", "collab"):
                assert getattr(r2, f).tobytes() == getattr(res, f).tobytes(), (s, f)
            sweep[s] = round(float(np.median(ts)), 6)
        piv = int(res.npiv.sum())
        a, b = float(np.median(ta)), float(np.median(tb))
        print(json.dumps({
            "workload": name, "lps": B, "n": n, "m": m, "cells": cells, "S": S,
            "pivots": piv, "status_counts": {int(k): int(v) for k, v in zip(*np.unique(res.status, return_counts=True))},
            "a_cluster_s": round(a, 6), "b_per_lp_s": round(b, 6), "a_reps_s": [round(t, 6) for t in ta],
            "b_reps_s": [round(t, 6) for t in tb],
            "a_lps_per_s": round(B / a, 1), "b_lps_per_s": round(B / b, 1),
            "a_pivots_per_s": round(piv / a), "b_pivots_per_s": round(piv / b),
            "a_cell_pivots_per_s": float(f"{piv * cells / a:.4g}"), "speedup": round(b / a, 2),
            "sweep_s_by_S": sweep, "bitwise_equal": True, "gpu": gpu,
            "torch": torch.__version__}), flush=True)


if __name__ == "__main__":
    main()
