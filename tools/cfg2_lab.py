#!/usr/bin/env python
"""Developer lab: cfg2 (1000 x 2000) full solve in each loop mode: pivots/s."""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from simplex_method_solver_b200 import workloads as W  # noqa: E402
from simplex_method_solver_b200.engine import DeviceTableau  # noqa: E402


def main():
    n, m = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (1000, 2000)
    rows, c = W.dense_lp(n, m, 0)
    modes = sys.argv[3].split(",") if len(sys.argv) > 3 else ["resident", "classic", "lookahead"]
    from simplex_method_solver_b200 import _native as N
    for mode in modes:
        tab = DeviceTableau(n, m, trace_capacity=200000)
        tab.load(rows, c, max_pivots=200000)
        tab.solve(stop_after=50, lookahead=mode)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st, npiv = tab.solve(chunk=256, lookahead=mode)
        e1.record()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        if os.environ.get("SPX_RESIDENT_STAMPS") and mode == "resident":
            import ctypes
            buf = (ctypes.c_uint64 * 16)()
            N.call("spx_resident_debug", buf)
            v = list(buf)
            piv = max(1, v[15])
            print("   cycles/pivot per phase (thread 0 of CTA 0, last launch, %d pivots): " % piv +
                  " ".join(f"[{k}]{v[k] / piv:.0f}" for k in range(15) if v[k]) + f"  sum {sum(v[:15]) / piv:.0f}")
        print(f"{n}x{m} {mode:10s}: status {st} npiv {npiv}  {ms:.1f} ms  {(npiv - 50) / ms * 1e3:.0f} pivots/s  "
              f"{ms / (npiv - 50) * 1e3:.2f} us/pivot (wall {dt * 1e3:.1f} ms)", flush=True)


if __name__ == "__main__":
    main()
