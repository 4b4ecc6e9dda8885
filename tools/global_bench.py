"""K8 (one cluster per LP, table in global memory) against the per-LP path, and against K7 where K7 fits.

(a) one ``solve_batched(tables, n, m, engine="global")`` call for the whole batch;
(b) one ``SimplexMethod(rows, c, engine="stream").solve()`` per LP (auto loop: the L2-resident kernel K5 at
    these sizes);
(c) on shapes K7 accepts, one ``solve_batched(..., engine="cluster")`` call.
All arms are warmed up, then run alternately --reps times in this process; end-to-end times are host clocks that
end in a device synchronise and include uploads and result downloads.  Kernel time is CUDA events around
``DeviceBatch.run()`` on an uploaded batch (re-uploaded before each timed run: K8 solves in place).  Every LP's
status, trace, final table, labels and x must be equal on every arm, and every forced cluster size that fits must
give (a)'s bits (the forced-size sweep records kernel time).  The co-resident working set is the tables of the
LPs whose clusters run at once.
Prints one JSON line per workload.

    python tools/global_bench.py [--reps 3] [--max-lps N] [--workloads d_600x800,...] [--no-per-lp] [--sweep-reps 1]
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

# name -> (LPs, generator, n, m, max_pivots).  The first four are above K7's capacity (n <= 528 at m = 800,
# m <= 9,499); the phase-1 1000 x 1000 family cycles, so its cap ends every LP; the last two are K7 shapes.
WORKLOADS = {
    "d_600x800": (64, W.dense_lp, 600, 800, 20000),
    "p1_1000x1000": (32, W.phase1_lp, 1000, 1000, 4000),
    "d_1000x2000": (16, W.dense_lp, 1000, 2000, 30000),
    "d_64x12000": (64, W.dense_lp, 64, 12000, 20000),
    "d_256x512": (64, W.dense_lp, 256, 512, 10000),
    "d_400x800": (16, W.dense_lp, 400, 800, 20000),
}
OPT_CLUSTER_SIZE = 16
L2_BYTES = 126 * 2**20
FIELDS = ("status", "npiv", "trace", "tables", "x", "obj", "rowlab", "collab")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def sync_time(fn):
    import torch
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def run_batch(tables, n, m, cap, engine):
    from simplex_method_solver_b200.batched import solve_batched
    return sync_time(lambda: solve_batched(tables, n, m, max_pivots=cap, engine=engine))


def run_per_lp(lps, cap):
    from simplex_method_solver_b200.simplex import SimplexMethod

    def go():
        out = []
        for rows, c in lps:
            sm = SimplexMethod(rows, c, engine="stream")
            out.append((sm.solve(max_pivots=cap), sm))
        return out
    return sync_time(go)


def kernel_times(tables, n, m, cap, reps):
    """CUDA-event time of DeviceBatch.run() (K8), one fresh upload before each run."""
    import torch
    from simplex_method_solver_b200.batched import DeviceBatch
    db = DeviceBatch(tables.shape[0], n, m, max_pivots=cap, engine="global")
    src = torch.from_numpy(tables).pin_memory()
    out = []
    for _ in range(reps + 1):
        db.upload(src)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        db.run()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / 1e3)
    return out[1:], db.cluster_size


def check_per_lp(res, outs):
    for k, (sol, sm) in enumerate(outs):
        assert int(res.status[k]) == sol.status and int(res.npiv[k]) == sol.npiv, k
        assert res.trace[k, : sol.npiv].tobytes() == np.ascontiguousarray(sol.trace, dtype=np.int32).tobytes(), k
        flat = np.concatenate([np.asarray(r, dtype=np.float64) for r in sm.table])
        assert res.tables[k].tobytes() == flat.tobytes(), k
        assert res.x[k].tobytes() == np.asarray(sol.x, dtype=np.float64).tobytes(), k


def check_same(r1, r2, what):
    for f in FIELDS:
        assert getattr(r1, f).tobytes() == getattr(r2, f).tobytes(), (what, f)


def forced_sizes(L, n, m):
    return [S for S in (1, 2, 4, 8, 16) if S >= L.spx_global_min_cluster_size(n, m)]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--max-lps", type=int, default=0, help="cap the LPs of every workload (0: as listed)")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--no-per-lp", action="store_true", help="skip arm (b)")
    ap.add_argument("--sweep-reps", type=int, default=1, help="timed kernel runs per forced cluster size")
    args = ap.parse_args()
    import torch
    from simplex_method_solver_b200 import _native as N
    L = N.lib()
    gpu = gpu_info()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    for name in args.workloads.split(","):
        B, gen, n, m, cap = WORKLOADS[name]
        if args.max_lps:
            B = min(B, args.max_lps)
        lps = [gen(n, m, seed) for seed in range(B)]
        tables = np.stack([np.concatenate([r.reshape(-1), c]) for r, c in lps])
        cells = n * (m + 1) + m
        k7 = L.spx_cluster_size(n, m) > 0
        S = L.spx_global_cluster_size(n, m, B)
        # warm-up of every arm
        run_batch(tables, n, m, cap, "global")
        if k7:
            run_batch(tables, n, m, cap, "cluster")
        if not args.no_per_lp:
            run_per_lp(lps[:2], cap)
        ta, tb, tc = [], [], []
        for _ in range(args.reps):
            t, res = run_batch(tables, n, m, cap, "global")
            ta.append(t)
            if not args.no_per_lp:
                t, outs = run_per_lp(lps, cap)
                tb.append(t)
            if k7:
                t, rc = run_batch(tables, n, m, cap, "cluster")
                tc.append(t)
        if not args.no_per_lp:
            check_per_lp(res, outs)
        if k7:
            check_same(res, rc, "cluster")
        kt, kS = kernel_times(tables, n, m, cap, args.reps)
        assert kS == S
        # forced cluster sizes: same bits, kernel time of each
        sweep_kernel = {}
        for s in forced_sizes(L, n, m):
            assert L.spx_set_option(OPT_CLUSTER_SIZE, s) == 0
            try:
                _, r2 = run_batch(tables, n, m, cap, "global")
                ks, _ = kernel_times(tables, n, m, cap, args.sweep_reps)
            finally:
                L.spx_set_option(OPT_CLUSTER_SIZE, 0)
            check_same(res, r2, f"S={s}")
            sweep_kernel[s] = round(float(np.median(ks)), 6)
        piv = int(res.npiv.sum())
        a, k = float(np.median(ta)), float(np.median(kt))
        # clusters the device runs at once at the default S (one 512-thread K8 CTA per SM), and their tables' bytes
        corun = min(B, max(1, sms // S))
        out = {
            "workload": name, "lps": B, "n": n, "m": m, "cells": cells, "max_pivots": cap, "S": S,
            "s_min": L.spx_global_min_cluster_size(n, m), "k7_fits": k7,
            "pivots": piv, "status_counts": {int(s): int(c) for s, c in zip(*np.unique(res.status, return_counts=True))},
            "a_global_s": round(a, 6), "a_reps_s": [round(t, 6) for t in ta],
            "a_kernel_s": round(k, 6), "a_kernel_reps_s": [round(t, 6) for t in kt],
            "a_lps_per_s": round(B / a, 1), "a_pivots_per_s": round(piv / a),
            "a_kernel_pivots_per_s": round(piv / k),
            "a_kernel_bytes_per_s": float(f"{16 * cells * piv / k:.4g}"),
            "corun_lps_at_S": corun, "corun_table_bytes": corun * cells * 8,
            "corun_fits_l2": corun * cells * 8 <= L2_BYTES,
            "sweep_kernel_s_by_S": sweep_kernel,
            "bitwise_equal": True, "gpu": gpu, "torch": torch.__version__}
        if tb:
            b = float(np.median(tb))
            out.update({"b_per_lp_s": round(b, 6), "b_reps_s": [round(t, 6) for t in tb],
                        "b_lps_per_s": round(B / b, 1), "b_pivots_per_s": round(piv / b),
                        "speedup_a_over_b": round(b / a, 2)})
        if tc:
            c = float(np.median(tc))
            out.update({"c_cluster_s": round(c, 6), "c_reps_s": [round(t, 6) for t in tc],
                        "c_lps_per_s": round(B / c, 1), "speedup_a_over_c": round(c / a, 2)})
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
