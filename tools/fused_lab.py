#!/usr/bin/env python
"""Developer lab: the F-pivots-per-pass fused loop on cfg4 (or --n/--m): pivots/s for each depth F,
with the pivot sequence checked against the golden prefix."""
import argparse
import json
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
    ap.add_argument("--pivots", type=int, default=400)
    ap.add_argument("--depths", default="1,2,4,8")
    ap.add_argument("--minb", default="3")
    ap.add_argument("--items", default="0", help="fused update kernel: column pairs per lane (0 = default, 1, 2)")
    ap.add_argument("--variants", default="0",
                    help="update kernel schedules as rows per warp strip, e.g. 0,32,64 (0 = the default)")
    a = ap.parse_args()
    L = N.lib()
    rows, c = W.dense_lp(a.n, a.m, 0)
    gold = None
    if (a.n, a.m) == (16384, 32768):
        with open(os.path.join(ROOT, "tests", "golden", "cfg_digests.json")) as fh:
            gold = np.asarray(json.load(fh)["cfg4"]["trace"], dtype=np.int32)
    cells = a.n * (a.m + 1) + a.m
    tab = DeviceTableau(a.n, a.m, trace_capacity=4 * a.pivots + 64)
    for mode, F, mb, trows, items in [("lookahead", 0, 0, 0, 0)] + [("fused", int(x), int(y), int(v), int(z))
                                                                    for v in a.variants.split(",")
                                                                    for z in a.items.split(",")
                                                                    for y in a.minb.split(",")
                                                                    for x in a.depths.split(",")]:
        if F:
            assert L.spx_set_option(N.OPT_FUSE_DEPTH, F) == 0
            assert L.spx_set_option(7, mb) == 0
            assert L.spx_set_option(11, trows) == 0
            assert L.spx_set_option(12, items) == 0
        tab.load(rows, c, max_pivots=4 * a.pivots + 32)
        tab.solve(stop_after=a.pivots, chunk=a.pivots, lookahead=mode)          # warm-up
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st, npiv = tab.solve(stop_after=a.pivots, chunk=a.pivots, lookahead=mode)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        ok = ""
        if gold is not None:
            tr = tab.trace[:npiv].cpu().numpy()
            k = min(len(gold), npiv)
            ok = f" golden[{k}]={'OK' if (tr[:k] == gold[:k]).all() else 'MISMATCH'}"
        print(f"{mode:9s} F={F} minb={mb} rows={trows} pairs={items}: {a.pivots} pivots in {ms:8.2f} ms  {a.pivots / ms * 1e3:8.1f} pivots/s  "
              f"{ms / a.pivots * 1e3:7.1f} us/pivot  north-star {16.0 * cells * a.pivots / ms / 1e6:8.0f} GB/s  "
              f"status={st} npiv={npiv}{ok}", flush=True)


if __name__ == "__main__":
    main()
