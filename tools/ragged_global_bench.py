"""Ragged batches that include LPs above K7's capacity: one solve_ragged(engine="auto_global") call against today's
practice of splitting the batch by hand, and the ragged K8 kernel against the uniform K8 kernel.

Mixed workload mixed_large (workloads.mixed_large_lps: mixed_lps(1024) at cap 20,000 plus 32 LPs above K7's capacity
at cap 4,000, 8 each of D(600,800), phase-1 1000 x 1000, D(2000,300), D(64,12000)):
  (a) one ``solve_ragged(lps, max_pivots=caps, engine="auto_global")`` call;
  (b) ``solve_ragged(engine="auto")`` on the LPs it accepts, plus one ``SimplexMethod(...).solve()`` per large LP;
  (c) ``solve_ragged(engine="auto")`` on the LPs it accepts, plus one ``solve_batched(engine="global")`` per large
      shape.
Uniform workloads (one shape, all on K8): CUDA-event kernel time of ``DeviceRaggedBatch.run`` (engine="global")
against ``DeviceBatch.run`` (engine="global") on the same uploaded batch (re-uploaded before each run: K8 solves in
place), both at the S each picks on the device.

End-to-end times are host clocks that end in a device synchronise and include packing, uploads and downloads.  Every
arm is warmed up, the arms alternate, and the median of --reps repetitions is reported.  Every LP's bits (status,
npiv, trace, final table, x, obj, labels) must be equal across the arms before a line is printed.  Prints one JSON
line per workload, with the GPU's name, power limit and maximum SM clock.

    python tools/ragged_global_bench.py [--reps 3] [--workloads mixed_large,u_600x800,u_p1_1000x1000]
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

# uniform workloads: name -> (LPs, generator, n, m, max_pivots)
UNIFORM = {
    "u_600x800": (64, W.dense_lp, 600, 800, 20000),
    "u_p1_1000x1000": (32, W.phase1_lp, 1000, 1000, 4000),
}
FIELDS = ("status", "npiv", "x", "obj", "tables", "rowlab", "collab", "trace")


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


def split(lps):
    """Indices of the LPs engine="auto" accepts, and the rest (above K7's capacity)."""
    from simplex_method_solver_b200.batched import kernel_for
    small, large = [], []
    for k, (rows, c) in enumerate(lps):
        (large if kernel_for(rows.shape[0], c.shape[0], "auto_global") == "global" else small).append(k)
    return small, large


def run_a(lps, caps):
    from simplex_method_solver_b200.batched import solve_ragged
    return sync_time(lambda: solve_ragged(lps, max_pivots=caps, engine="auto_global"))


def run_b(lps, caps, small, large):
    from simplex_method_solver_b200.batched import solve_ragged
    from simplex_method_solver_b200.simplex import SimplexMethod

    def go():
        rs = solve_ragged([lps[k] for k in small], max_pivots=[caps[k] for k in small])
        out = []
        for k in large:
            sm = SimplexMethod(*lps[k], engine="stream")
            out.append((sm.solve(max_pivots=caps[k]), sm))
        return rs, out
    return sync_time(go)


def run_c(lps, caps, small, large):
    from simplex_method_solver_b200.batched import solve_batched, solve_ragged

    def go():
        rs = solve_ragged([lps[k] for k in small], max_pivots=[caps[k] for k in small])
        groups = {}
        for k in large:
            groups.setdefault((lps[k][0].shape[0], lps[k][1].shape[0], caps[k]), []).append(k)
        out = {}
        for (n, m, cap), idx in groups.items():
            tables = np.stack([np.concatenate([lps[k][0].reshape(-1), lps[k][1]]) for k in idx])
            out[(n, m, cap)] = (idx, solve_batched(tables, n, m, max_pivots=cap, engine="global"))
        return rs, out
    return sync_time(go)


def check_small(ra, rs, small):
    for j, k in enumerate(small):
        for f, a, b in zip(rs.lp(j)._fields, ra.lp(k), rs.lp(j)):
            if a is not None:
                assert a.tobytes() == b.tobytes(), (k, f)


def check_b(ra, out, large):
    for k, (sol, sm) in zip(large, out):
        one = ra.lp(k)
        assert int(one.status[0]) == sol.status and int(one.npiv[0]) == sol.npiv, k
        assert one.trace[0, : sol.npiv].tobytes() == np.ascontiguousarray(sol.trace, dtype=np.int32).tobytes(), k
        assert one.tables[0].tobytes() == sm._dev.export_flat(sm._npiv).tobytes(), k
        assert one.x[0].tobytes() == np.asarray(sol.x, dtype=np.float64).tobytes(), k
        assert float(one.obj[0]).hex() == float(sol.obj2).hex(), k
        assert one.rowlab[0].tolist() == list(sol.rowlab) and one.collab[0].tolist() == list(sol.collab), k


def check_c(ra, out):
    for idx, res in out.values():
        for j, k in enumerate(idx):
            one = ra.lp(k)
            for f in FIELDS:
                assert getattr(one, f).tobytes() == getattr(res, f)[j: j + 1].tobytes(), (k, f)


def median(v):
    return round(float(np.median(v)), 6)


def mixed_large(reps, gpu, torch_version):
    from simplex_method_solver_b200.batched import DeviceRaggedBatch, pack_ragged
    lps, caps = W.mixed_large_lps(1024, 0)
    small, large = split(lps)
    run_a(lps, caps)                                        # warm-up of every arm (b: two of its large LPs)
    run_b(lps, caps, small, large[:2])
    run_c(lps, caps, small, large)
    ta, tb, tc = [], [], []
    for _ in range(reps):
        t, ra = run_a(lps, caps)
        ta.append(t)
        t, (rsb, outb) = run_b(lps, caps, small, large)
        tb.append(t)
        t, (rsc, outc) = run_c(lps, caps, small, large)
        tc.append(t)
    check_small(ra, rsb, small)
    check_small(ra, rsc, small)
    check_b(ra, outb, large)
    check_c(ra, outc)
    shapes, _ = pack_ragged(lps)
    db = DeviceRaggedBatch(shapes, caps, engine="auto_global")
    launches = [{"kind": la["kind"], "planned_S": la["S"], "S": S, "lps": int(len(la["lps"]))}
                for la, S in zip(db.plan.launches, db.cluster_sizes)]
    a, b, c = median(ta), median(tb), median(tc)
    print(json.dumps({
        "workload": "mixed_large", "lps": len(lps), "large_lps": len(large),
        "shapes": int(len({tuple(s) for s in shapes.tolist()})), "launches": launches,
        "pivots": int(ra.npiv.sum()), "large_pivots": int(ra.npiv[large].sum()),
        "status_counts": {int(k): int(v) for k, v in zip(*np.unique(ra.status, return_counts=True))},
        "a_one_call_s": a, "b_auto_plus_per_lp_s": b, "c_auto_plus_per_shape_s": c,
        "speedup_a_over_b": round(b / a, 2), "speedup_a_over_c": round(c / a, 3),
        "a_reps_s": [round(t, 6) for t in ta], "b_reps_s": [round(t, 6) for t in tb],
        "c_reps_s": [round(t, 6) for t in tc],
        "bitwise_equal": True, "gpu": gpu, "torch": torch_version}), flush=True)


def uniform(name, reps, gpu, torch_version):
    import torch
    from simplex_method_solver_b200.batched import DeviceBatch, DeviceRaggedBatch
    B, gen, n, m, cap = UNIFORM[name]
    lps = [gen(n, m, s) for s in range(B)]
    tables = np.stack([np.concatenate([r.reshape(-1), c]) for r, c in lps])
    src = torch.from_numpy(tables).pin_memory()
    flat = src.reshape(-1)
    dr = DeviceRaggedBatch([(n, m)] * B, cap, engine="global")
    du = DeviceBatch(B, n, m, max_pivots=cap, engine="global")

    def timed(db, data):
        db.upload(data)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        db.run()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / 1e3
    timed(dr, flat), timed(du, src)                         # warm-up
    kr, ku = [], []
    for _ in range(reps):
        kr.append(timed(dr, flat))
        ku.append(timed(du, src))
    rr, ru = dr.result(), du.result()
    for k in range(B):
        one = rr.lp(k)
        for f in FIELDS:
            assert getattr(one, f).tobytes() == getattr(ru, f)[k: k + 1].tobytes(), (k, f)
    piv = int(rr.npiv.sum())
    print(json.dumps({
        "workload": name, "lps": B, "n": n, "m": m, "max_pivots": cap, "pivots": piv,
        "ragged_S": dr.cluster_sizes[0], "uniform_S": du.cluster_size,
        "ragged_kernel_s": median(kr), "uniform_kernel_s": median(ku),
        "kernel_ragged_over_uniform": round(float(np.median(kr) / np.median(ku)), 3),
        "ragged_kernel_reps_s": [round(t, 6) for t in kr], "uniform_kernel_reps_s": [round(t, 6) for t in ku],
        "bitwise_equal": True, "gpu": gpu, "torch": torch_version}), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--workloads", default="mixed_large," + ",".join(UNIFORM))
    args = ap.parse_args()
    import torch
    from simplex_method_solver_b200 import _native as N
    N.lib()
    gpu = gpu_info()
    for name in args.workloads.split(","):
        if name == "mixed_large":
            mixed_large(args.reps, gpu, torch.__version__)
        else:
            uniform(name, args.reps, gpu, torch.__version__)


if __name__ == "__main__":
    main()
