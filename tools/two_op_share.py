"""Share of the levels of cfg4's one-GPU fused passes whose cells take the two-operation quotient (two_op_flag in
csrc/spx_fused.cu): runs pivots [0, warmup + steps) x 1000 of cfg4 as passes of 16 levels, reads each pass's plan
flags, and prints one JSON line for the pivots bench.py times (after its warm-up) and one for all of them.

    python tools/two_op_share.py [--warmup 3] [--steps 5]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from simplex_method_solver_b200 import workloads as W  # noqa: E402
from simplex_method_solver_b200.engine import DeviceTableau  # noqa: E402

N_ROWS, M_COLS, SEED, DEPTH = 16384, 32768, 0, 16
TWO_OFFSET = 640          # byte offset of SoloPlan::two in the plan at the start of the workspace (static_assert there)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    rows, c = W.dense_lp(N_ROWS, M_COLS, SEED)
    need = (args.warmup + args.steps) * 1000
    tab = DeviceTableau(N_ROWS, M_COLS, device=dev, trace_capacity=need + 64)
    tab.load(rows, c, max_pivots=need + 64)
    words = tab.work.view(torch.int32)
    per_level = []                                           # (pivot index, flag)
    full_passes = passes = 0
    while len(per_level) < need:
        tab.fused_pass(DEPTH, 0)
        head = words[: (TWO_OFFSET // 4) + DEPTH].cpu()
        f = int(head[0])
        assert f == DEPTH, f
        two = head[TWO_OFFSET // 4:].tolist()
        per_level += [(len(per_level) + k, two[k]) for k in range(f)]
        passes += 1
        full_passes += all(two[:f])
    timed = [t for i, t in per_level if args.warmup * 1000 <= i < need]
    print(json.dumps({"workload": "cfg4", "pivots": f"[{args.warmup * 1000}, {need})", "levels": len(timed),
                      "two_op_share": sum(timed) / len(timed), "card": torch.cuda.get_device_name(0)}))
    print(json.dumps({"workload": "cfg4", "pivots": f"[0, {need})", "levels": len(per_level),
                      "two_op_share": sum(t for _, t in per_level) / len(per_level),
                      "passes_all_levels_two_op": full_passes / passes, "passes": passes}))


if __name__ == "__main__":
    main()
