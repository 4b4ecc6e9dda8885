"""Ragged batches (one solve_ragged call for LPs of mixed shapes) against today's per-shape practice.

Mixed workloads (gui_ragged: 10 shapes, all K4 warp mode; mixed_lps: hundreds of shapes over every class):
  (a) one ``solve_ragged(lps, max_pivots=cap)`` call;
  (b) group the LPs by (n, m, cap) and make one ``solve_batched`` call per group.
Uniform workloads (one shape; the cost of the ragged machinery itself): the ragged entry against the uniform
entry on the same batch.

End-to-end times are host clocks that end in a device synchronise and include packing, uploads and downloads;
kernel times are CUDA events around ``DeviceRaggedBatch.run`` / the ``DeviceBatch.run`` calls, with the tables
uploaded before the first event.  For the mixed workloads each class of the plan (warp mode, CTA mode, each
cluster size) is also timed alone, so the idle tail between the sequential class launches shows as the
difference between the whole run and the sum of its classes.  Every arm is warmed up, the arms alternate, and
the median of --reps repetitions is reported.  Every LP's bits (status, npiv, trace, final table, x, obj,
labels) must be equal across the arms before a line is printed.  Prints one JSON line per workload.

    python tools/ragged_bench.py [--reps 5] [--workloads gui_ragged,mixed_lps,cfg3,km10,p1_100x100,d_128x256]
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


def _uniform(B, gen):
    return lambda: [gen(s) for s in range(B)]


# name -> (kind, LPs generator, max_pivots)
WORKLOADS = {
    "gui_ragged": ("mixed", lambda: W.gui_ragged(65536, 0), 64),
    "mixed_lps": ("mixed", lambda: W.mixed_lps(4096, 0), 20000),
    "cfg3": ("uniform", lambda: [(T, C) for T, C in zip(*W.gui_batch(65536, 0))], 64),
    "km10": ("uniform", _uniform(1024, lambda s: W.klee_minty(10)), 1024),
    "p1_100x100": ("uniform", _uniform(1024, lambda s: W.phase1_lp(100, 100, s)), 2000),
    "d_128x256": ("uniform", _uniform(256, lambda s: W.dense_lp(128, 256, s)), 4000),
}
FIELDS = ("status", "npiv", "x", "obj", "tables", "rowlab", "collab", "trace")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def sync():
    import torch
    torch.cuda.synchronize()


def groups_of(lps, cap):
    """(n, m, cap) -> ([LP indices], [B, cells] tables): today's practice."""
    g = {}
    for k, (rows, c) in enumerate(lps):
        g.setdefault((rows.shape[0], c.shape[0], cap), []).append(k)
    return {key: (idx, np.stack([np.concatenate([lps[k][0].reshape(-1), lps[k][1]]) for k in idx]))
            for key, idx in g.items()}


def run_a(lps, cap):
    from simplex_method_solver_b200.batched import solve_ragged
    t0 = time.perf_counter()
    res = solve_ragged(lps, max_pivots=cap)
    sync()
    return time.perf_counter() - t0, res


def uniform_engine(n, m):
    """spx_solve_batched cannot launch K4 CTA-mode shapes of more than 48 KB of shared memory (it asks for 227 KB of
    dynamic shared memory on top of the kernel's static bytes): today such a group has to go to K7 (same bits)."""
    cells = n * (m + 1) + m
    lut = (cells * 4 + 15) // 16 * 16
    wb = ((2 * cells + m) * 8 + (n + m) * 4 + 15) // 16 * 16
    return "cluster" if 96 < cells <= 10000 and lut + wb > 48 * 1024 else "auto"


def run_b(lps, cap):
    from simplex_method_solver_b200.batched import solve_batched
    t0 = time.perf_counter()
    out = {}
    for (n, m, c), (idx, tables) in groups_of(lps, cap).items():
        out[(n, m, c)] = (idx, solve_batched(tables, n, m, max_pivots=c, engine=uniform_engine(n, m)))
    sync()
    return time.perf_counter() - t0, out


def check_equal(ra, rb):
    for idx, res in rb.values():
        for j, k in enumerate(idx):
            one = ra.lp(k)
            for f in FIELDS:
                a, b = getattr(one, f), getattr(res, f)[j: j + 1]
                assert a.tobytes() == b.tobytes(), (k, f)


def event_time(fn, prepare):
    """CUDA-event time (s) of fn() after prepare() (not timed)."""
    import torch
    prepare()
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / 1e3


def ragged_kernel_time(shapes, packed, cap):
    from simplex_method_solver_b200.batched import DeviceRaggedBatch
    db = DeviceRaggedBatch(shapes, cap)
    return lambda: event_time(db.run, lambda: db.upload(packed)), db


def grouped_kernel_time(lps, cap):
    from simplex_method_solver_b200.batched import DeviceBatch
    dbs = [(DeviceBatch(len(idx), n, m, c, engine=uniform_engine(n, m)), tables)
           for (n, m, c), (idx, tables) in groups_of(lps, cap).items()]

    def prepare():
        for db, tables in dbs:
            db.upload(tables)

    def run():
        for db, _ in dbs:
            db.run()
    return lambda: event_time(run, prepare), len(dbs)


def median(v):
    return round(float(np.median(v)), 6)


def mixed(name, lps, cap, reps, gpu, torch_version):
    from simplex_method_solver_b200.batched import pack_ragged
    shapes, packed = pack_ragged(lps)
    run_a(lps, cap)                                         # warm-up of both arms
    run_b(lps, cap)
    ta, tb = [], []
    for _ in range(reps):
        t, ra = run_a(lps, cap)
        ta.append(t)
        t, rb = run_b(lps, cap)
        tb.append(t)
    check_equal(ra, rb)
    ka_fn, db = ragged_kernel_time(shapes, packed, cap)
    kb_fn, ngroups = grouped_kernel_time(lps, cap)
    ka_fn(), kb_fn()
    ka, kb = [], []
    for _ in range(reps):
        ka.append(ka_fn())
        kb.append(kb_fn())
    # each class of the plan alone: the same launch the whole plan makes for it
    per_class = []
    for la in db.plan.launches:
        idx = np.sort(la["lps"])
        sub = [lps[k] for k in idx]
        s_shapes, s_packed = pack_ragged(sub)
        fn, sdb = ragged_kernel_time(s_shapes, s_packed, cap)
        assert sdb.launches == 1
        fn()
        per_class.append({"kind": la["kind"], "S": la["S"], "lps": int(len(idx)), "threads": la["threads"],
                          "smem": la["smem"], "kernel_s": median([fn() for _ in range(reps)])})
    piv = int(ra.npiv.sum())
    a, b = median(ta), median(tb)
    print(json.dumps({
        "workload": name, "lps": len(lps), "shapes": int(len({tuple(s) for s in shapes.tolist()})), "groups": ngroups,
        "b_groups_sent_to_k7": sum(uniform_engine(int(n), int(m)) == "cluster" for n, m in {tuple(s) for s in shapes.tolist()}),
        "launches": db.launches, "max_pivots": cap, "pivots": piv,
        "status_counts": {int(k): int(v) for k, v in zip(*np.unique(ra.status, return_counts=True))},
        "a_ragged_s": a, "b_grouped_s": b, "speedup": round(b / a, 2),
        "a_reps_s": [round(t, 6) for t in ta], "b_reps_s": [round(t, 6) for t in tb],
        "a_kernel_s": median(ka), "b_kernel_s": median(kb), "kernel_speedup": round(float(np.median(kb) / np.median(ka)), 2),
        "a_lps_per_s": round(len(lps) / a, 1), "b_lps_per_s": round(len(lps) / b, 1),
        "per_class_kernel": per_class, "sum_of_classes_s": round(sum(c["kernel_s"] for c in per_class), 6),
        "bitwise_equal": True, "gpu": gpu, "torch": torch_version}), flush=True)


def uniform(name, lps, cap, reps, gpu, torch_version):
    from simplex_method_solver_b200.batched import DeviceBatch, pack_ragged, solve_batched
    n, m = lps[0][0].shape[0], lps[0][1].shape[0]
    tables = np.stack([np.concatenate([r.reshape(-1), c]) for r, c in lps])

    def run_u():
        t0 = time.perf_counter()
        res = solve_batched(tables, n, m, max_pivots=cap)
        sync()
        return time.perf_counter() - t0, res
    run_a(lps, cap)
    run_u()
    ta, tu = [], []
    for _ in range(reps):
        t, ra = run_a(lps, cap)
        ta.append(t)
        t, ru = run_u()
        tu.append(t)
    check_equal(ra, {(n, m, cap): (list(range(len(lps))), ru)})
    shapes, packed = pack_ragged(lps)
    ka_fn, db = ragged_kernel_time(shapes, packed, cap)
    du = DeviceBatch(len(lps), n, m, cap)
    ku_fn = lambda: event_time(du.run, lambda: du.upload(tables))  # noqa: E731
    ka_fn(), ku_fn()
    ka, ku = [], []
    for _ in range(reps):
        ka.append(ka_fn())
        ku.append(ku_fn())
    a, u = median(ta), median(tu)
    print(json.dumps({
        "workload": name, "lps": len(lps), "n": n, "m": m, "kernel": db.plan.launches[0]["kind"],
        "S": db.plan.launches[0]["S"], "max_pivots": cap, "pivots": int(ra.npiv.sum()),
        "ragged_s": a, "uniform_s": u, "ragged_over_uniform": round(a / u, 3),
        "ragged_kernel_s": median(ka), "uniform_kernel_s": median(ku),
        "kernel_ragged_over_uniform": round(float(np.median(ka) / np.median(ku)), 3),
        "ragged_kernel_reps_s": [round(t, 6) for t in ka], "uniform_kernel_reps_s": [round(t, 6) for t in ku],
        "bitwise_equal": True, "gpu": gpu, "torch": torch_version}), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    import torch
    from simplex_method_solver_b200 import _native as N
    N.lib()
    for name in args.workloads.split(","):
        kind, gen, cap = WORKLOADS[name]
        lps = gen()
        gpu = gpu_info()
        (mixed if kind == "mixed" else uniform)(name, lps, cap, args.reps, gpu, torch.__version__)


if __name__ == "__main__":
    main()
