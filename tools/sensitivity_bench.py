"""The sensitivity kernels (csrc/spx_sensitivity.cu) against the bytes of the final tables they read.

Workloads, each solved first (to optimality where the cap allows):
  u_k4      4,096 D(20, 20)         uniform, K4 (DeviceBatch, engine="auto_global")
  u_k7      256 phase-1 128 x 256   uniform, K7
  u_k8      64 D(600, 800)          uniform, K8 (3.8 MB per table)
  mixed     workloads.mixed_large_lps(1024): a ragged batch over K4, K7 and K8 (DeviceRaggedBatch, "auto_global")
  split     D(1000, 2000) solved by SimplexMethod.solve() to optimality (the split layout)
For each: the CUDA-event time of the report's launches (spx_sensitivity_*, outputs preallocated, median of --reps
windows of --iters calls after a warm-up), the table bytes one pass reads, the bytes/s that makes, and the time of
the solve it follows.  The report's outputs are checked bit for bit against tests/sensitivity_oracle.c on a sample
of LPs before a line is printed.  Prints one JSON line per workload with the GPU's name, power limit and maximum SM
clock.  The tables of u_k8 and mixed (246 MB and about 600 MB) exceed the 126 MB L2; the others are read from L2
after the first call.

    python tools/sensitivity_bench.py [--reps 5] [--iters 20] [--workloads u_k4,u_k7,u_k8,mixed,split]
"""
from __future__ import annotations

import argparse
import ctypes
import importlib.util
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from simplex_method_solver_b200 import workloads as W  # noqa: E402

UNIFORM = {"u_k4": (4096, W.dense_lp, 20, 20, 5000), "u_k7": (256, W.phase1_lp, 128, 256, 5000),
           "u_k8": (64, W.dense_lp, 600, 800, 20000)}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def oracle_module():
    spec = importlib.util.spec_from_file_location("sensitivity_oracle", os.path.join(ROOT, "tests", "sensitivity_oracle.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def same(got, want):
    for g, w in zip(got, want):
        g, w = np.asarray(g, dtype=np.float64), np.asarray(w, dtype=np.float64).reshape(np.shape(g))
        assert (np.isnan(g) == np.isnan(w)).all() and g[~np.isnan(g)].tobytes() == w[~np.isnan(w)].tobytes()


def event_time(fn, reps, iters):
    import torch
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) / 1e3 / iters)
    return float(np.median(ts))


def sync_time(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def report(name, kernel_s, table_bytes, solve_s, optimal, B):
    print(json.dumps({"workload": name, "gpu": gpu_info(), "lps": B, "optimal": int(optimal),
                      "table_bytes": int(table_bytes), "sensitivity_kernel_s": kernel_s,
                      "table_GB_per_s": table_bytes / kernel_s / 1e9, "solve_s": solve_s,
                      "share_of_solve": kernel_s / solve_s, "bits_checked": True}), flush=True)


def run_uniform(name, reps, iters, SO):
    import torch
    from simplex_method_solver_b200 import _native as N
    from simplex_method_solver_b200.batched import DeviceBatch, _SensOut
    B, gen, n, m, cap = UNIFORM[name]
    tabs = np.stack([np.concatenate([r.reshape(-1), c]) for r, c in (gen(n, m, s) for s in range(B))])
    db = DeviceBatch(B, n, m, max_pivots=cap, trace=False, engine="auto_global")
    db.upload(tabs)
    solve_s, _ = sync_time(db.run)
    res, rep = db.result(), db.sensitivity()
    for k in range(0, B, max(1, B // 16)):
        same([a[k] for a in rep[:5]], SO.sensitivity(res.tables[k], n, m, res.rowlab[k], res.collab[k], res.status[k] == 0))
    out = _SensOut(B * n, B * m, db.device)
    stream = torch.cuda.current_stream().cuda_stream
    fn = lambda: N.call("spx_sensitivity_batched", db.T.data_ptr(), B, n, m, db.status.data_ptr(),  # noqa: E731
                        db.rowlab.data_ptr(), db.collab.data_ptr(), *out.ptrs(), stream)
    report(f"{name}:{db.kernel}", event_time(fn, reps, iters), 8 * B * db.cells, solve_s, rep.optimal.sum(), B)


def run_mixed(reps, iters, SO):
    import torch
    from simplex_method_solver_b200 import _native as N
    from simplex_method_solver_b200.batched import DeviceRaggedBatch, _SensOut, pack_ragged
    lps, caps = W.mixed_large_lps(1024)
    shapes, packed = pack_ragged(lps)
    db = DeviceRaggedBatch(shapes, caps, trace=False, engine="auto_global")
    db.upload(packed)
    solve_s, _ = sync_time(db.run)
    res, rep = db.result(), db.sensitivity()
    for k in list(range(0, db.B, 64)) + list(range(db.B - 32, db.B, 4)):
        one, n, m = res.lp(k), int(shapes[k, 0]), int(shapes[k, 1])
        same([a[0] for a in rep.lp(k)[:5]], SO.sensitivity(one.tables[0], n, m, one.rowlab[0], one.collab[0],
                                                           one.status[0] == 0))
    out = _SensOut(db.totals[2], db.totals[1], db.device)
    stream = torch.cuda.current_stream().cuda_stream
    fn = lambda: N.call("spx_sensitivity_ragged", db.T.data_ptr(), db.plan.plan.ctypes.data,  # noqa: E731
                        db.d_plan.data_ptr(), db.status.data_ptr(), db.rowlab.data_ptr(), db.collab.data_ptr(),
                        *out.ptrs(), stream)
    report("mixed_large", event_time(fn, reps, iters), 8 * db.totals[0], solve_s, rep.optimal.sum(), db.B)


def run_split(reps, iters, SO):
    import torch
    from simplex_method_solver_b200 import _native as N
    from simplex_method_solver_b200.batched import _SensOut
    from simplex_method_solver_b200.simplex import SimplexMethod
    n, m = 1000, 2000
    rows, c = W.dense_lp(n, m, 0)
    sm = SimplexMethod(rows, c)
    solve_s, sol = sync_time(sm.solve)
    assert sol.status == 0
    rep = sm.sensitivity()
    rl, cl = sm._dev.labels_host()
    same(rep[:5], SO.sensitivity(sm._dev.export_flat(sm._npiv), n, m, rl, cl, True))
    dev, cur = sm._dev, sm._dev.cur(sm._npiv)
    out = _SensOut(n, m, dev.device)
    opt = ctypes.c_int32(0)
    stream = torch.cuda.current_stream().cuda_stream
    fn = lambda: N.call("spx_sensitivity_split", dev.A[cur].data_ptr(), dev.b[cur].data_ptr(), n, m, dev.ld,  # noqa: E731
                        dev.rowlab.data_ptr(), dev.collab.data_ptr(), *out.ptrs(), ctypes.byref(opt), stream)
    # the split entry synchronises once per call (its optimality test reads b and the f row on the host)
    report("split_D1000x2000", event_time(fn, reps, iters), 8 * (n * (m + 1) + m), solve_s, 1, 1)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--workloads", default="u_k4,u_k7,u_k8,mixed,split")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sensitivity_bench.py needs a CUDA device")
    SO = oracle_module()
    for w in a.workloads.split(","):
        if w in UNIFORM:
            run_uniform(w, a.reps, a.iters, SO)
        elif w == "mixed":
            run_mixed(a.reps, a.iters, SO)
        elif w == "split":
            run_split(a.reps, a.iters, SO)
        else:
            raise SystemExit(f"unknown workload {w!r}")


if __name__ == "__main__":
    main()
