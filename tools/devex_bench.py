"""The three entering rules of the batched engines on the GPU: pivots, kernel time and end-to-end time per rule, one
JSON line per (workload, rule), then one line per workload with devex's kernel time per pivot over Dantzig's.

  a  1,024 scaled phase1_lp(100, 100) LPs on K7 at S = 1 (SPX_OPT_CLUSTER_SIZE = 1)
  b  64 scaled D(256, 512) on K7 (its default S)
  c  16 scaled D(600, 800) on K8 (its default S)
  d  workloads.scaled_lps(4096) through solve_ragged(engine="auto_global")
  e  workloads.mixed_lps(4096), the unscaled control, the same way
"Scaled": column j of an LP and c_j times 10^U(-2, 2), a change of the units of x_j (workloads.scaled_lps).

kernel_ms: CUDA events around the solve's launches on resident buffers (best of --reps, after one warm-up run of
the same launches).  e2e_ms: host clock around solve_batched / solve_ragged (upload, launches, result copy, which
synchronises), best of --reps.  Every LP gets the cap --cap.  The card's name and power limit are read in the same
call.  Usage: python tools/devex_bench.py [--only abcde] [--reps 3] [--cap 200000] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from simplex_method_solver_b200 import batched as Bt  # noqa: E402
from simplex_method_solver_b200 import _native as N  # noqa: E402
from simplex_method_solver_b200 import workloads as W  # noqa: E402

RULES = ("reference", "dantzig", "devex")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def scale(rows, c, seed):
    s = 10.0 ** np.random.default_rng(seed + 7).uniform(-2.0, 2.0, c.shape[0])
    rows = rows.copy()
    rows[:, : c.shape[0]] *= s
    return rows, c * s


def workloads():
    """name -> (kind, payload, engine, forced cluster size)"""
    def flats(lps):
        return np.stack([np.concatenate([r.reshape(-1), c]) for r, c in lps])
    return {
        "a": ("uniform", (flats([scale(*W.phase1_lp(100, 100, s), s) for s in range(1024)]), 100, 100), "cluster", 1),
        "b": ("uniform", (flats([scale(*W.dense_lp(256, 512, s), s) for s in range(64)]), 256, 512), "cluster", 0),
        "c": ("uniform", (flats([scale(*W.dense_lp(600, 800, s), s) for s in range(16)]), 600, 800), "global", 0),
        "d": ("ragged", W.scaled_lps(4096, 0), "auto_global", 0),
        "e": ("ragged", W.mixed_lps(4096, 0), "auto_global", 0),
    }


def events(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def leg(kind, payload, engine, rule, cap, reps):
    code = N.RULES[rule]
    if kind == "uniform":
        T, n, m = payload
        db = Bt.DeviceBatch(T.shape[0], n, m, max_pivots=cap, trace=False, engine=engine)

        def load():
            db.upload(T)

        def e2e():
            return Bt.solve_batched(T, n, m, max_pivots=cap, rule=rule, trace=False, engine=engine)
    else:
        shapes, packed = Bt.pack_ragged(payload)
        db = Bt.DeviceRaggedBatch(shapes, max_pivots=cap, trace=False, engine=engine)

        def load():
            db.upload(packed)

        def e2e():
            return Bt.solve_ragged(payload, max_pivots=cap, rule=rule, trace=False, engine=engine)
    kernel = []
    for q in range(reps + 1):                  # the first run loads the kernels
        load()
        torch.cuda.synchronize()
        t = events(lambda: db.run(code))
        if q:
            kernel.append(t)
    res = db.result()
    wall = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = e2e()
        torch.cuda.synchronize()
        wall.append((time.perf_counter() - t0) * 1e3)
    assert np.array_equal(r.npiv, res.npiv) and np.array_equal(r.status, res.status)
    return {"pivots": int(res.npiv.astype(np.int64).sum()), "max_lp_pivots": int(res.npiv.max()),
            "optimal": int((res.status == N.OPTIMAL).sum()), "capped": int((res.status == N.CAP).sum()),
            "lps": int(res.status.shape[0]), "kernel_ms": min(kernel), "e2e_ms": min(wall)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="abcde")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cap", type=int, default=200000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.init()
    gpu = card()
    out = open(a.out, "a") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()
    L = N.lib()
    for name, (kind, payload, engine, S) in workloads().items():
        if name not in a.only:
            continue
        got = {}
        assert L.spx_set_option(N.OPT_CLUSTER_SIZE, S) == 0
        try:
            for rule in RULES:
                got[rule] = leg(kind, payload, engine, rule, a.cap, a.reps)
                emit({"workload": name, "rule": rule, **got[rule], "gpu": gpu})
        finally:
            L.spx_set_option(N.OPT_CLUSTER_SIZE, 0)
        per = {r: got[r]["kernel_ms"] / max(got[r]["pivots"], 1) for r in RULES}
        emit({"workload": name, "devex_over_dantzig_kernel_ms_per_pivot": per["devex"] / per["dantzig"],
              "dantzig_over_devex_pivots": got["dantzig"]["pivots"] / max(got["devex"]["pivots"], 1),
              "dantzig_over_devex_kernel_ms": got["dantzig"]["kernel_ms"] / got["devex"]["kernel_ms"],
              "gpu": gpu})


if __name__ == "__main__":
    main()
