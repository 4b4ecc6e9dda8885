"""The four entering rules of the batched engines on the GPU, Dantzig with Bland's rule on degenerate pivots
(rule="dantzig_bland") against the three that keep the reference's phase 1: pivots, LPs that end at the cap, kernel
time and end-to-end time per rule, one JSON line per (workload, rule), then one line per workload comparing
dantzig_bland with Dantzig.

  p  32 phase1_lp(1000, 1000) on K8 (its default S), cap 20,000: the phase-1 family that cycles under the other rules
  m  workloads.mixed_lps(4096) through solve_ragged(engine="auto_global"), cap 50,000
  s  workloads.scaled_lps(4096) the same way, cap 50,000
  d  64 D(256, 512) on K7 (its default S), cap 50,000: non-degenerate, so the rule's price per pivot shows

kernel_ms: CUDA events around the solve's launches on resident buffers (best of --reps, after one warm-up run of
the same launches).  e2e_ms: host clock around solve_batched / solve_ragged (upload, launches, result copy, which
synchronises), best of --reps.  The card's name and power limit are read in the same call.
Usage: python tools/dantzig_bland_bench.py [--only pmsd] [--reps 2] [--out FILE]
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

RULES = ("reference", "dantzig", "devex", "dantzig_bland")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def workloads():
    """name -> (kind, payload, engine, cap)"""
    def flats(lps):
        return np.stack([np.concatenate([r.reshape(-1), c]) for r, c in lps])
    return {
        "p": ("uniform", (flats([W.phase1_lp(1000, 1000, s) for s in range(32)]), 1000, 1000), "global", 20000),
        "m": ("ragged", W.mixed_lps(4096, 0), "auto_global", 50000),
        "s": ("ragged", W.scaled_lps(4096, 0), "auto_global", 50000),
        "d": ("uniform", (flats([W.dense_lp(256, 512, s) for s in range(64)]), 256, 512), "cluster", 50000),
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
    ap.add_argument("--only", default="pmsd")
    ap.add_argument("--reps", type=int, default=2)
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
    for name, (kind, payload, engine, cap) in workloads().items():
        if name not in a.only:
            continue
        got = {}
        for rule in RULES:
            got[rule] = leg(kind, payload, engine, rule, cap, a.reps)
            emit({"workload": name, "rule": rule, "cap": cap, **got[rule], "gpu": gpu})
        per = {r: got[r]["kernel_ms"] / max(got[r]["pivots"], 1) for r in RULES}
        emit({"workload": name,
              "dantzig_bland_over_dantzig_kernel_ms_per_pivot": per["dantzig_bland"] / per["dantzig"],
              "dantzig_over_dantzig_bland_kernel_ms": got["dantzig"]["kernel_ms"] / got["dantzig_bland"]["kernel_ms"],
              "gpu": gpu})
    emit({"card_after": card()})


if __name__ == "__main__":
    main()
