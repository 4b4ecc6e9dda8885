#!/usr/bin/env python
"""Record tests/golden/fresh_cases.json: the outcomes tests/test_oracle.py compares the oracle with on its seeded
"fresh" LPs (the inputs are not those of reference_cases.json):

  families  150 LPs per family (gui2dp / smallint / dense), cap 60   -> test_oracle_equals_live_reference
  medium    dense_lp(60, 90, 5), 25 pivots, every pivot and table    -> test_oracle_pick_update_equal_live_reference_medium
  sharded   util.make_lp families of the sharded-flow tests          -> test_oracle_equals_live_reference_on_the_sharded_test_lps
  dantzig   90 LPs under the Dantzig entering rule, cap 150          -> test_dantzig_rule_equals_reference_driven_by_column_swap

    SIMPLEX_REF=<original project>/src python tests/golden/make_fresh_cases.py    # provenance "reference"
    python tests/golden/make_fresh_cases.py                                       # provenance "oracle"

With $SIMPLEX_REF the original's own simplex.py computes every outcome (driven as in make_golden.py).  Without it the
oracle (oracle/spx_oracle.c) does, and the file says so; the tests then pin the oracle to that record, and check the
record against the original on any run where $SIMPLEX_REF is set.
"""
from __future__ import annotations

import importlib.util
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.dirname(HERE)):
    sys.path.insert(0, p)

import oracle  # noqa: E402
from simplex_method_solver_b200 import workloads as W  # noqa: E402
from util import (FRESH_SHARDED_LPS, drive_reference, flat_of, fresh_dantzig_lps, fresh_lps, make_lp,  # noqa: E402
                  table_sha)

STATUS_TO_END = {0: "optimal", -1: "incorrect system", -2: "simplex method does not converge", -3: "cap"}


def load_reference():
    src = os.environ.get("SIMPLEX_REF", "")
    if not src:
        return None, None
    sys.path.insert(0, src)
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)                          # imports the original's simplex.py from $SIMPLEX_REF
    return mg.ref, mg


def record(rows, c, cap, ref, labels=True):
    m = rows.shape[1] - 1
    if ref is not None:
        end, trace, flat, rl, cl = drive_reference(ref, rows, c, cap)
    else:
        o = oracle.solve(rows, c, max_pivots=cap)
        end, trace, flat = STATUS_TO_END[o.status], o.trace.tolist(), o.table
        rl, cl = oracle.label_strings(o.rowlab, o.collab, m)
    out = {"end": end, "trace": trace, "table_sha256": table_sha(flat)}
    if labels:
        out["row_labels"], out["column_labels"] = list(rl), list(cl)
    return out


def medium(ref):
    n, m, k = 60, 90, 25
    rows, c = W.dense_lp(n, m, 5)
    pivots = []
    if ref is not None:
        sm = ref.SimplexMethod(rows.tolist(), c.tolist())
        for _ in range(k):
            ok, i, j, e = sm.pick_element()
            assert ok
            sm.recalculate_matrix()
            pivots.append([i, j, float(e).hex(), table_sha(np.asarray([v for row in sm.table for v in row]))])
    else:
        T = flat_of(rows, c)
        for _ in range(k):
            st, i, j, e = oracle.pick(T, n, m)
            assert st == oracle.PIVOT
            T = oracle.update(T, n, m, i, j)
            pivots.append([i, j, float(e).hex(), table_sha(T)])
    return {"n": n, "m": m, "seed": 5, "pivots": pivots}


def dantzig(ref, mg):
    out = []
    for rows, c in fresh_dantzig_lps():
        if ref is not None:
            sm, trace, end, _ = mg.drive_dantzig(rows.tolist(), c.tolist(), 150)
            out.append({"end": end, "trace": trace, "table_sha256": mg.table_sha(sm.table)})
        else:
            o = oracle.solve(rows, c, max_pivots=150, rule="dantzig")
            out.append({"end": STATUS_TO_END[o.status], "trace": o.trace.tolist(), "table_sha256": table_sha(o.table)})
    return out


def main():
    ref, mg = load_reference()
    doc = {"made_by": "tests/golden/make_fresh_cases.py",
           "provenance": "reference" if ref is not None else "oracle",
           "families": {f: [record(rows, c, 60, ref) for rows, c in fresh_lps(f)] for f in ("gui2dp", "smallint", "dense")},
           "medium": medium(ref),
           "sharded": [dict(record(*make_lp(n, m, 7, kind), cap, ref), n=n, m=m, cap=cap, kind=kind)
                       for n, m, cap, kind in FRESH_SHARDED_LPS],
           "dantzig": dantzig(ref, mg)}
    with open(os.path.join(HERE, "fresh_cases.json"), "w") as fh:
        json.dump(doc, fh, separators=(",", ":"))
        fh.write("\n")
    print("fresh_cases.json:", doc["provenance"], os.path.getsize(os.path.join(HERE, "fresh_cases.json")), "bytes")


if __name__ == "__main__":
    main()
