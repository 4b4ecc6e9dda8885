#!/usr/bin/env python
"""Developer lab: time every schedule of the K3 update kernel (occupancy target, tile height) on
one tableau shape and check that all schedules write bit-identical output.  Runs on a GPU box:

    python tools/upd_lab.py [--n 16384 --m 32768 --reps 20]

Prints one line per schedule: mean/min CUDA-event time per launch and the algorithmic GB/s
(16 B x cells / time).  Not part of the product path or the test-suite.
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from simplex_method_solver_b200 import _native as N  # noqa: E402
from simplex_method_solver_b200 import workloads as W  # noqa: E402
from simplex_method_solver_b200.engine import DeviceTableau  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--m", type=int, default=32768)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--variants", default="")
    args = ap.parse_args()
    n, m = args.n, args.m
    L = N.lib()
    rows, c = W.dense_lp(n, m, 0)
    tab = DeviceTableau(n, m)
    tab.load(rows, c, max_pivots=1 << 40)
    del rows
    cells = n * (m + 1) + m
    variants = [
        ("tiled minb=2", {2: 2, 5: 0}),
        ("tiled minb=3", {2: 3, 5: 0}),
        ("tiled minb=4", {2: 4, 5: 0}),
        ("tiled minb=3 tr=32", {2: 3, 5: 32}),
        ("tiled minb=3 tr=16", {2: 3, 5: 16}),
        ("tiled minb=3 tr=8", {2: 3, 5: 8}),
        ("tiled minb=4 tr=16", {2: 4, 5: 16}),
        ("tiled minb=4 tr=8", {2: 4, 5: 8}),
    ]
    if args.variants:
        keep = set(args.variants.split(","))
        variants = [v for k, v in enumerate(variants) if str(k) in keep]
    # one real pivot decision; every variant applies the same pivot from buffer 0 to buffer 1
    tab.pick(0)
    st0 = tab.read_state()
    assert st0.status == N.PIVOT
    ref = None
    for name, opts in variants:
        for k, v in opts.items():
            assert L.spx_set_option(k, v) == 0
        times = []
        for rep in range(args.reps + 3):
            tab.write_state(st0)                       # npiv stays 0: the update is re-applied
            # L2 is far smaller than the 8.6 GB streamed per launch: no flush needed for cfg4;
            # for small shapes flush with a 256 MB write
            if cells * 16 < (512 << 20):
                torch.empty(64 << 20, dtype=torch.float32, device="cuda").zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            tab.update(0)
            e1.record()
            torch.cuda.synchronize()
            if rep >= 3:
                times.append(e0.elapsed_time(e1))
        out = tab.A[1]
        if ref is None:
            ref = out.clone()
            bref = tab.b[1].clone()
            same = True
        else:
            same = bool(torch.equal(out.view(torch.int64), ref.view(torch.int64))
                        and torch.equal(tab.b[1].view(torch.int64), bref.view(torch.int64)))
        st = tab.read_state()
        mean, best = float(np.mean(times)), float(np.min(times))
        print(f"{name:24s} mean {mean:8.4f} ms  min {best:8.4f} ms  {16.0 * cells / mean / 1e6:8.1f} GB/s "
              f"(best {16.0 * cells / best / 1e6:8.1f})  identical={same} npiv={st.npiv} "
              f"hints=({st.hint_bneg[1]},{st.hint_fneg[1]})", flush=True)
    # back-to-back sustained: 100 launches of the auto choice, ping-ponging
    for name, opts in variants:
        for k, v in opts.items():
            L.spx_set_option(k, v)
        tab.write_state(st0)
        for _ in range(10):
            tab.write_state(st0); tab.update(0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        K = 100
        e0.record()
        for _ in range(K):
            L.spx_update(tab.A[0].data_ptr(), tab.A[1].data_ptr(), tab.b[0].data_ptr(), tab.b[1].data_ptr(),
                         n, m, tab.ld, tab.state.data_ptr(), tab.colbuf.data_ptr(), tab.rowlab.data_ptr(),
                         tab.collab.data_ptr(), None, torch.cuda.current_stream().cuda_stream)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / K
        print(f"sustained {name:24s} {ms:8.4f} ms/launch  {16.0 * cells / ms / 1e6:8.1f} GB/s", flush=True)


if __name__ == "__main__":
    main()
