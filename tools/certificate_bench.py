"""The certificate kernels (csrc/spx_certificate.cu): CUDA-event time of the report against the bytes it reads.

Workloads:
  cfg3      the 1,048,576 GUI-like 8 x 2 LPs of bench.py's cfg3 leg (W.gui_batch(1 << 20, 0)) after a K4 solve
  mixed     workloads.mixed_lps(4096) as one ragged batch (DeviceRaggedBatch, "auto_global", cap 20,000)
  split     a failed 16384 x 32768 split table: D(16384, 32768) with b < 0 in every tenth row (each of them with
            positive cells) and row 16383 turned into a Farkas row (b < 0, A <= 0), as SimplexMethod holds it
For each: the time of one report (spx_certificate_*, outputs preallocated, median of --reps windows of --iters calls
after a warm-up), the bytes a report must read (b, the f row and the labels of every LP, and every cell of every
candidate row and column: an upper bound on the cells the tile pass reads), and that over the time as a share of
the 6,538 GB/s copy peak bench.py uses.  The outputs are checked bit for bit against tests/certificate_oracle.c on
a sample of LPs before a line is printed.  Prints one JSON line per workload with the GPU's name, power limit and
maximum SM clock.

    python tools/certificate_bench.py [--reps 5] [--iters 20] [--workloads cfg3,mixed,split]
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from simplex_method_solver_b200 import workloads as W  # noqa: E402

COPY_PEAK = 6538e9        # bytes/s: the measured copy_ peak bench.py reports against


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def oracle_module():
    spec = importlib.util.spec_from_file_location("certificate_oracle",
                                                  os.path.join(ROOT, "tests", "certificate_oracle.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def same(got, want):
    assert (int(got[0]), int(got[3])) == (want[0], want[3])
    for k in (1, 2, 4, 5):
        g, w = np.asarray(got[k], dtype=np.float64), np.asarray(want[k], dtype=np.float64).reshape(np.shape(got[k]))
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


def needed_bytes(T, n, m):
    """bytes the reports of LPs T [B, cells] (or one LP [cells]) must read: b, f, labels, and the cells of the
    candidate rows and columns"""
    T = np.asarray(T).reshape(-1, n * (m + 1) + m)
    w = m + 1
    b, f = T[:, m: n * w: w], T[:, n * w: n * w + m]
    rows = np.sum(np.isfinite(b) & (b < 0), axis=1)
    cols = np.sum(np.isfinite(f) & (f < 0), axis=1) * np.all(np.isfinite(b) & (b >= 0), axis=1)
    return int(np.sum(12 * (n + m) + 8 * (rows * m + cols * n)))


def report(name, kernel_s, nbytes, B, cert):
    print(json.dumps({"workload": name, "gpu": gpu_info(), "lps": B, "infeasible": int(np.sum(cert[0] >= 0)),
                      "unbounded": int(np.sum(cert[3] >= 0)), "bytes_needed": int(nbytes),
                      "certificate_kernel_s": kernel_s, "GB_per_s": nbytes / kernel_s / 1e9,
                      "share_of_copy_peak": nbytes / kernel_s / COPY_PEAK, "bits_checked": True}), flush=True)


def run_cfg3(reps, iters, CO):
    import torch
    from simplex_method_solver_b200 import _native as N
    from simplex_method_solver_b200.batched import DeviceBatch, _CertOut
    B, n, m = 1 << 20, 8, 2
    T, C = W.gui_batch(B, 0)
    tabs = W.batch_flat(T, C)
    db = DeviceBatch(B, n, m, max_pivots=64, trace=False)
    db.upload(tabs)
    db.run()
    res, cert = db.result(), db.certificate()
    for k in range(0, B, B // 64):
        same([a[k] for a in cert[1:4] + cert[5:]], CO.certificate(res.tables[k], n, m, res.rowlab[k], res.collab[k]))
    nbytes = needed_bytes(res.tables, n, m)
    out = _CertOut(B, B * n, B * m, db.device)
    stream = torch.cuda.current_stream().cuda_stream
    fn = lambda: N.call("spx_certificate_batched", db.T.data_ptr(), B, n, m, db.rowlab.data_ptr(),  # noqa: E731
                        db.collab.data_ptr(), *out.ptrs(), stream)
    report("cfg3_1048576x(8x2)", event_time(fn, reps, iters), nbytes, B, (cert.farkas_row, 0, 0, cert.ray_col))


def run_mixed(reps, iters, CO):
    import torch
    from simplex_method_solver_b200 import _native as N
    from simplex_method_solver_b200.batched import DeviceRaggedBatch, _CertOut, pack_ragged
    lps = W.mixed_lps(4096)
    shapes, packed = pack_ragged(lps)
    db = DeviceRaggedBatch(shapes, 20000, trace=False, engine="auto_global")
    db.upload(packed)
    db.run()
    res, cert = db.result(), db.certificate()
    nbytes = 0
    for k in range(db.B):
        one, n, m = res.lp(k), int(shapes[k, 0]), int(shapes[k, 1])
        nbytes += needed_bytes(one.tables[0], n, m)
        if k % 64 == 0:
            c = cert.lp(k)
            same([a[0] for a in c[1:4] + c[5:]], CO.certificate(one.tables[0], n, m, one.rowlab[0], one.collab[0]))
    out = _CertOut(db.B, db.totals[2], db.totals[1], db.device)
    stream = torch.cuda.current_stream().cuda_stream
    fn = lambda: N.call("spx_certificate_ragged", db.T.data_ptr(), db.plan.plan.ctypes.data,  # noqa: E731
                        db.d_plan.data_ptr(), db.rowlab.data_ptr(), db.collab.data_ptr(), *out.ptrs(), stream)
    report("mixed_lps_4096", event_time(fn, reps, iters), nbytes, db.B, (cert.farkas_row, 0, 0, cert.ray_col))


def run_split(reps, iters, CO):
    import torch
    from simplex_method_solver_b200 import _native as N
    from simplex_method_solver_b200.batched import _CertOut
    from simplex_method_solver_b200.simplex import SimplexMethod
    n, m = 16384, 32768
    rows, c = W.dense_lp(n, m, 0)
    rows[::10, m] = -rows[::10, m]               # candidate rows; D's cells are all negative, so give each a positive
    rows[::10, 7] = 1.0
    rows[n - 1] = -np.abs(rows[n - 1])           # the Farkas row
    sm = SimplexMethod(rows, c, engine="stream")
    del rows
    cert = sm.certificate()
    dev, cur = sm._dev, sm._dev.cur(sm._npiv)
    flat = dev.export_flat(sm._npiv)
    rl, cl = dev.labels_host()
    same([cert.farkas_row, cert.farkas, cert.farkas_bound, cert.ray_col, cert.ray, cert.ray_slope],
         CO.certificate(flat, n, m, rl, cl))
    assert cert.farkas_row == n - 1
    nbytes = needed_bytes(flat, n, m)
    del flat
    out = _CertOut(1, n, m, dev.device)
    stream = torch.cuda.current_stream().cuda_stream
    fn = lambda: N.call("spx_certificate_split", dev.A[cur].data_ptr(), dev.b[cur].data_ptr(), n, m, dev.ld,  # noqa: E731
                        dev.rowlab.data_ptr(), dev.collab.data_ptr(), *out.ptrs(), stream)
    report("split_failed_16384x32768", event_time(fn, reps, iters), nbytes, 1,
           (np.array([cert.farkas_row]), 0, 0, np.array([cert.ray_col])))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--workloads", default="cfg3,mixed,split")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("certificate_bench.py needs a CUDA device")
    CO = oracle_module()
    runs = {"cfg3": run_cfg3, "mixed": run_mixed, "split": run_split}
    for w in a.workloads.split(","):
        if w not in runs:
            raise SystemExit(f"unknown workload {w!r}")
        runs[w](a.reps, a.iters, CO)


if __name__ == "__main__":
    main()
