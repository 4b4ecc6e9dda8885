"""Warm start against cold solves on the GPU: device-event kernel times and pivots per LP, one JSON line per leg.

  continue  64 x phase1_lp(600, 800) on K8: one solve at cap C against a solve at C/2 plus a resume of C/2
  cost      4,096 x D(20, 20) on K4 and 64 x D(600, 800) on K8, costs scaled by 1 +- U(0, 5 %): a cold solve of the
            new LPs against change + resume from the optimal final tables
  rhs       the same LPs, one right-hand side per LP moved by half ("inside") and by 1.5 times ("beyond") its
            sensitivity range toward its finite end
  change    the change kernel alone on the 64 x D(600, 800) tables, every delta nonzero: the bytes the statement reads
            and writes over the kernel time, as a share of the 7.7 TB/s data-sheet HBM figure of one B200

The card's name and power limit are read in the same call.  Usage: python tools/warm_bench.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from simplex_method_solver_b200 import batched as Bt  # noqa: E402
from simplex_method_solver_b200 import _native as N  # noqa: E402
from simplex_method_solver_b200 import workloads as W  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fn, reps=2):
    """best of reps device-event times of fn() in ms: the kernels fn launches on the current stream"""
    best = float("inf")
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def warm_up(tabs, n, m, engine):
    """load every kernel a leg times (solve, change, resume) before its timed launches"""
    r = Bt.solve_batched(tabs[:1], n, m, max_pivots=1, engine=engine)
    Bt.resolve(r, tabs[:1], rhs=tabs[:1, m: n * (m + 1): m + 1] + 1.0, cost=tabs[:1, n * (m + 1):] * 2,
               max_pivots=1, engine=engine)
    torch.cuda.synchronize()


def batch(lps):
    return np.stack([np.concatenate([r.reshape(-1), c]) for r, c in lps])


def leg_continue(out):
    n, m, B, C = 600, 800, 64, 2000
    tabs = batch([W.phase1_lp(n, m, s) for s in range(B)])
    fn = tabs[:, n * (m + 1):]
    warm_up(tabs, n, m, "global")
    full = Bt.DeviceBatch(B, n, m, max_pivots=C, trace=False, engine="global")
    half = Bt.DeviceBatch(B, n, m, max_pivots=C // 2, trace=False, engine="global")
    full.upload(tabs)
    t_full = timed(lambda: full.run(), reps=1)
    rf = full.result()
    half.upload(tabs)
    t_first = timed(lambda: half.run(), reps=1)
    t_resume = timed(lambda: half.resume(fn), reps=1)
    rs = half.result()
    out({"leg": "continue", "lps": B, "shape": [n, m], "cap": C, "cold_kernel_ms": t_full,
         "split_kernel_ms": t_first + t_resume, "resume_kernel_ms": t_resume,
         "same_tables": bool(rf.tables.tobytes() == rs.tables.tobytes()),
         "pivots_per_lp": float(rf.npiv.mean())})


def cost_and_rhs(out, n, m, B, engine, seed):
    g = np.random.default_rng(seed)
    lps = [W.dense_lp(n, m, seed + s) for s in range(B)]
    tabs = batch(lps)
    warm_up(tabs, n, m, engine)
    cap = 20000
    base = Bt.DeviceBatch(B, n, m, max_pivots=cap, trace=False, engine=engine)
    base.upload(tabs)
    base.run()
    r0 = base.result()
    rep = base.sensitivity()
    c0 = tabs[:, n * (m + 1):]
    b0 = tabs[:, : n * (m + 1)].reshape(B, n, m + 1)[:, :, m]
    cost = c0 * (1 + g.uniform(-0.05, 0.05, (B, m)))
    legs = [("cost", None, cost)]
    for name, f in (("rhs_inside", 0.5), ("rhs_beyond", 1.5)):
        rhs = b0.copy()
        for q in range(B):
            fin = [(k, s) for k in range(n) for s in (0, 1) if np.isfinite(rep.rhs_range[q, k, s]) and rep.rhs_range[q, k, s] > 0]
            if fin:
                k, s = fin[g.integers(len(fin))]
                rhs[q, k] += (1 if s else -1) * f * rep.rhs_range[q, k, s]
        legs.append((name, rhs, None))
    for name, rhs, cst in legs:
        new = tabs.copy()
        if cst is not None:
            new[:, n * (m + 1):] = cst
        if rhs is not None:
            new[:, m: n * (m + 1): m + 1] = rhs       # the b cell of each row
        cold = Bt.DeviceBatch(B, n, m, max_pivots=cap, trace=False, engine=engine)
        cold.upload(new)
        t_cold = timed(lambda: cold.run(), reps=1)
        rc = cold.result()
        warm = Bt.DeviceBatch(B, n, m, max_pivots=cap, trace=False, engine=engine)
        db = None if rhs is None else rhs - b0
        dc = None if cst is None else cst - c0
        fnew = c0 if cst is None else cst

        warm.upload(r0.tables)
        warm.upload_labels(r0.rowlab, r0.collab)
        d_db = None if db is None else torch.from_numpy(np.ascontiguousarray(db)).cuda()
        d_dc = None if dc is None else torch.from_numpy(np.ascontiguousarray(dc)).cuda()
        stream = torch.cuda.current_stream().cuda_stream
        t_change = timed(lambda: N.call("spx_warm_change_batched", warm.T.data_ptr(), B, n, m, warm.rowlab.data_ptr(),
                                        warm.collab.data_ptr(), N.ptr(d_db), N.ptr(d_dc), stream), reps=1)
        t_resume = timed(lambda: warm.resume(fnew), reps=1)    # (includes the [B, m] upload of the new costs)
        rw = warm.result()
        both = (rc.status == 0) & (rw.status == 0)
        out({"leg": name, "lps": B, "shape": [n, m], "engine": engine, "cold_kernel_ms": t_cold,
             "change_kernel_ms": t_change, "resume_ms": t_resume, "warm_ms": t_change + t_resume,
             "cold_pivots_per_lp": float(rc.npiv.mean()), "warm_pivots_per_lp": float(rw.npiv.mean()),
             "optimal_cold": int((rc.status == 0).sum()), "optimal_warm": int((rw.status == 0).sum()),
             "max_rel_obj_diff": float(np.max(np.abs(rc.obj[both] - rw.obj[both]) / (1 + np.abs(rc.obj[both]))))
             if both.any() else None})
    return r0, tabs


def leg_change(out, r0, n, m):
    B = r0.status.shape[0]
    g = np.random.default_rng(1)
    db, dc = g.uniform(0.5, 1.0, (B, n)), g.uniform(0.5, 1.0, (B, m))
    dv = Bt.DeviceBatch(B, n, m, max_pivots=0, trace=False, engine="global")
    dv.upload(r0.tables)
    dv.upload_labels(r0.rowlab, r0.collab)
    dv.change(db, dc)
    torch.cuda.synchronize()
    reps = 20
    t = timed(lambda: [dv.change(db, dc) for _ in range(reps)]) / reps     # includes the two delta uploads
    d_db, d_dc = torch.from_numpy(db).cuda(), torch.from_numpy(dc).cuda()
    s = torch.cuda.current_stream().cuda_stream
    k = lambda: N.call("spx_warm_change_batched", dv.T.data_ptr(), B, n, m, dv.rowlab.data_ptr(),  # noqa: E731
                       dv.collab.data_ptr(), d_db.data_ptr(), d_dc.data_ptr(), s)
    tk = timed(lambda: [k() for _ in range(reps)]) / reps
    yb = (r0.rowlab >= m).sum(axis=1)               # active columns of the b update
    xr = (r0.collab < m).sum(axis=1)                # active rows of the f update
    cells_read = (n * (yb + 1) + m * (xr + 1)).sum()
    nbytes = 8 * cells_read + 8 * B * (n + m) * 2 + 4 * B * (n + m) + 8 * B * (n + m)
    out({"leg": "change", "lps": B, "shape": [n, m], "kernel_ms": tk, "with_upload_ms": t,
         "bytes": int(nbytes), "bytes_per_s": nbytes / (tk * 1e-3),
         "share_of_7.7TBps": nbytes / (tk * 1e-3) / HBM_BYTES_PER_S})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rows = []
    c = card()

    def out(d):
        d["card"] = c
        print(json.dumps(d), flush=True)
        rows.append(d)
    leg_continue(out)
    cost_and_rhs(out, 20, 20, 4096, "smem", 100)
    r0, _ = cost_and_rhs(out, 600, 800, 64, "global", 200)
    leg_change(out, r0, 600, 800)
    if a.out:
        with open(a.out, "w") as fh:
            for d in rows:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
