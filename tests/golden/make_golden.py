#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/ by RUNNING THE REFERENCE.

Run with $SIMPLEX_REF pointing at the original project's src/ directory:

    SIMPLEX_REF=<original project>/src python tests/golden/make_golden.py [small] [cfg2] [cfg3] [cfg5] [cfg4]

The reference's solver (its src/simplex.py) is stdlib-only, so it is
imported and driven with its own pick_element() / recalculate_matrix() /
get_solution().  Every fixture records its provenance:

  "reference" — produced by the live reference itself;
  "oracle"    — produced by oracle/spx_oracle.c (for sizes the pure-Python
                reference cannot reach), which tests/test_oracle.py checks
                bit-for-bit against every "reference" fixture.

The reference's sources are not part of this repository; the tests read only
these JSON files (and the reference too where $SIMPLEX_REF is set).
Floats are stored as float.hex() strings so fixtures are bit-exact.
"""
from __future__ import annotations

import hashlib
import json
import os
import struct
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF_SRC = os.environ.get("SIMPLEX_REF", "")
if not REF_SRC:
    raise SystemExit("set SIMPLEX_REF to the original project's src/ directory")
sys.path.insert(0, REF_SRC)

import simplex as ref  # noqa: E402  (the reference)

from simplex_method_solver_b200 import workloads as W  # noqa: E402


def hx(v):
    return float(v).hex()


def drive(rows, c, cap):
    """The reference's own manual driving pattern (simplex.py:261-269)."""
    sm = ref.SimplexMethod([[float(v) for v in r] for r in rows], [float(v) for v in c])
    trace = []
    try:
        while True:
            ok, i, j, e = sm.pick_element()
            if not ok:
                return sm, trace, "optimal", (i, j, e)
            if len(trace) >= cap:
                return sm, trace, "cap", None
            trace.append([i, j])
            sm.recalculate_matrix()
    except ValueError as e:
        return sm, trace, str(e), None


def table_hex(table):
    return [[hx(v) for v in row] for row in table]


def table_sha(table):
    h = hashlib.sha256()
    for row in table:
        for v in row:
            h.update(struct.pack("<d", float(v)))
    return h.hexdigest()


def case(name, rows, c, cap=200, snapshots=False):
    sm, trace, end, fin = drive(rows, c, cap)
    out = {
        "name": name, "provenance": "reference",
        "rows": [[hx(v) for v in r] for r in rows], "c": [hx(v) for v in c],
        "cap": cap, "end": end, "trace": trace,
        "final_table": table_hex(sm.table), "final_table_sha256": table_sha(sm.table),
        "row_labels": list(sm.row), "column_labels": list(sm.column),
    }
    if fin is not None:
        out["x1"], out["x2"], out["f"] = hx(fin[0]), hx(fin[1]), hx(fin[2])
    if snapshots and end != "cap":
        res = ref.SimplexMethod([[float(v) for v in r] for r in rows],
                                [float(v) for v in c]).get_solution()
        snaps = []
        for it in res:
            if isinstance(it, ref.Error):
                snaps.append({"error": str(it)})
            else:
                snaps.append({"row": it.row, "column": it.column, "table": table_hex(it.table),
                              "i": it.i, "j": it.j, "x1": hx(it.x1), "x2": hx(it.x2),
                              "optimum": hx(it.optimum)})
        out["get_solution"] = snaps
        out["snapshot_sha256"] = W.snapshot_digest(
            [it.table for it in res if not isinstance(it, ref.Error)])
    return out


def make_small():
    cases = []
    # the reference's own examples: simplex.py:205-229 (commented) and :231-238 (demos)
    cases.append(case("ref_example_cfg1_205", W.CFG1_ROWS, W.CFG1_C, snapshots=True))
    cases.append(case("ref_example_210",
                      [[12.50, -26.60, 726.78], [-26.40, -18.40, 1814.48], [-6, 41.80, -81.00],
                       [22.30, 16.20, -780.76], [17.50, -3.60, -105.43]], [2.4, -1.15],
                      snapshots=True))
    cases.append(case("ref_example_216_noconv",
                      [[-39.00, 93.10, 113.10], [-45.50, 89.90, 250.25], [-45.50, 67.00, 441.35],
                       [-45.50, 47.20, 746.20], [-45.50, 24.90, 1392.30],
                       [-45.50, 12.90, 1810.90], [-45.50, 45.50, -45.50]], [-1, -2.45],
                      snapshots=True))
    cases.append(case("ref_example_224_incorrect", [[-1.00, -1.00, -1]], [-1, 0], snapshots=True))
    cases.append(case("ref_example_226",
                      [[-45.50, 12.20, 1810.90], [-44.20, 56.30, -73.19],
                       [2.50, -92.60, 3764.32]], [-1, -2.45], snapshots=True))
    cases.append(case("ref_demo_231", [[1, 1, -2], [-1, 1, 1.5], [1, -2, 4]], [-1, -1],
                      snapshots=True))
    cases.append(case("ref_demo_235", [[1, 1, -2], [-1, 1, 2], [0, -1, 2]], [-1, 0],
                      snapshots=True))
    # quirks of the selection rules (SURVEY.md §3.3 / G-quirks)
    cases.append(case("quirk_first_negative_entering", [[-1, -1, 10]], [-1, -5], snapshots=True))
    cases.append(case("quirk_tie_last_row", [[-1, 0, 5], [-2, 0, 10], [-1, 0, 5]], [-1, 0],
                      snapshots=True))
    cases.append(case("quirk_max_negative_ratio", [[-1, 0, 5], [-1, 0, 3], [-2, 0, 6], [-1, 0, 4]],
                      [-1, 0], snapshots=True))
    cases.append(case("quirk_zero_then_negative", [[-1, 0, 0], [-1, 0, 5]], [-1, 0],
                      snapshots=True))
    cases.append(case("quirk_cycles_forever", [[1, 0, 3], [2, 0, 0]], [-1, 0], cap=25))
    cases.append(case("quirk_unbounded_noconv", [[1, 0, 3], [2, 0, 1]], [-1, 0], snapshots=True))
    cases.append(case("quirk_phase1_then_incorrect", [[1, 1, -2], [-1, -1, 1]], [1, 1],
                      snapshots=True))
    cases.append(case("quirk_negative_zero_b", [[-1, -1, -0.0], [-1, 1, 4]], [-1, -1],
                      snapshots=True))
    cases.append(case("quirk_already_optimal", [[-1, -1, 4]], [1, 1], snapshots=True))
    cases.append(case("quirk_zero_column_skipped", [[0, -1, 4], [-1, 0, 3], [0, 0, 1]], [-1, -1],
                      snapshots=True))
    cases.append(case("quirk_wide_m5", [[-1, -2, -3, -1, -2, 30], [-2, -1, -1, -3, -1, 40],
                                        [1, 0, 0, 0, 0, -1]], [-1, -1, -2, -1, -3],
                      snapshots=True))
    # random families (SURVEY.md Appendix A), n in [1,9], m in [2,6], cap 200
    rng = np.random.default_rng(20261018)
    for t in range(360):
        n = int(rng.integers(1, 10))
        m = int(rng.integers(2, 7))
        fam = t % 3
        if fam == 0:
            A = np.round(rng.uniform(-50, 50, (n, m)), 2)
            b = np.round(rng.uniform(-500, 2000, n), 2)
            c = np.round(rng.uniform(-3, 3, m), 2)
        elif fam == 1:
            A = rng.integers(-3, 4, (n, m)).astype(float)
            b = rng.integers(-2, 7, n).astype(float)
            c = rng.integers(-3, 4, m).astype(float)
        else:
            A = -rng.uniform(0.1, 1, (n, m))
            b = rng.uniform(1, 2, n)
            c = -rng.uniform(0.1, 1, m)
        rows = np.hstack([A, b[:, None]]).tolist()
        cc = case(f"random_{['gui2dp', 'smallint', 'dense'][fam]}_{t:03d}", rows, c.tolist(), cap=200)
        del cc["final_table"]          # keep the fixture small: digest only
        cases.append(cc)
    # a few mid-size LPs the reference still solves in seconds
    for (n, m, seed) in [(30, 40, 1), (64, 33, 2), (17, 96, 3)]:
        rows, c = W.dense_lp(n, m, seed)
        cc = case(f"dense_{n}x{m}_seed{seed}", rows.tolist(), c.tolist(), cap=5000)
        del cc["final_table"]
        del cc["rows"], cc["c"]
        cc["generator"] = {"kind": "dense_lp", "n": n, "m": m, "seed": seed}
        cases.append(cc)
    with open(os.path.join(HERE, "reference_cases.json"), "w") as fh:
        json.dump({"made_by": "tests/golden/make_golden.py small",
                   "reference": "jqnfxa/Simplex-Method-Solver src/simplex.py",
                   "cases": cases}, fh, indent=0)
    ends = {}
    for cc in cases:
        ends[cc["end"]] = ends.get(cc["end"], 0) + 1
    print("small:", len(cases), "cases", ends)


def load_cfg():
    p = os.path.join(HERE, "cfg_digests.json")
    if os.path.exists(p):
        with open(p) as fh:
            return json.load(fh)
    return {"made_by": "tests/golden/make_golden.py"}


def save_cfg(d):
    with open(os.path.join(HERE, "cfg_digests.json"), "w") as fh:
        json.dump(d, fh, indent=1, sort_keys=True)


def make_cfg2():
    import oracle
    d = load_cfg()
    rows, c = W.dense_lp(1000, 2000, 0)
    out = {"generator": {"kind": "dense_lp", "n": 1000, "m": 2000, "seed": 0},
           "input_sha256": W.input_digest(rows, c)}
    # the reference itself: first 12 pivots (1.3 s each) + tableau digest after them
    t0 = time.time()
    sm, trace, end, _ = drive(rows.tolist(), c.tolist(), cap=12)
    out["reference_first12"] = {"provenance": "reference", "trace": trace,
                                "table_sha256_after12": table_sha(sm.table),
                                "seconds": round(time.time() - t0, 2)}
    # the oracle: full run
    s = oracle.solve(rows, c, max_pivots=200000)
    tr = s.trace
    out["oracle_full"] = {
        "provenance": "oracle", "status": int(s.status), "npiv": int(s.npiv),
        "pivot_sha256_after100": W.pivot_digest(tr[:100]),
        "pivot_sha256_after1000": W.pivot_digest(tr[:1000]),
        "pivot_sha256_final": W.pivot_digest(tr),
        "table_sha256_after12": hashlib.sha256(
            oracle.solve(rows, c, max_pivots=12).table.tobytes()).hexdigest(),
        "final_table_sha256": hashlib.sha256(s.table.tobytes()).hexdigest(),
        "objm": hx(s.objm), "obj2": hx(s.obj2),
        "x_sha256": hashlib.sha256(s.x.astype("<f8").tobytes()).hexdigest(),
        "x_first8": [hx(v) for v in s.x[:8]],
        "collab_sha256": hashlib.sha256(s.collab.astype("<i4").tobytes()).hexdigest(),
        "rowlab_sha256": hashlib.sha256(s.rowlab.astype("<i4").tobytes()).hexdigest(),
    }
    d["cfg2"] = out
    save_cfg(d)
    print("cfg2:", out["reference_first12"]["trace"], out["oracle_full"]["npiv"])


def make_cfg3():
    d = load_cfg()
    B = 65536
    T, C = W.gui_batch(B, 0)
    out = {"generator": {"kind": "gui_batch", "B": B, "seed": 0},
           "input_sha256": W.input_digest(T, C), "provenance": "reference"}
    h_p, h_s = hashlib.sha256(), hashlib.sha256()
    hist, ends = {}, {}
    first = []
    t0 = time.time()
    for k in range(B):
        sm, trace, end, fin = drive(T[k].tolist(), C[k].tolist(), cap=1000)
        ends[end] = ends.get(end, 0) + 1
        hist[len(trace)] = hist.get(len(trace), 0) + 1
        for (r, c) in trace:
            h_p.update(struct.pack("<iii", k, r, c))
        x1, x2, f = fin if fin is not None else (float("nan"),) * 3
        h_s.update(struct.pack("<ddd", x1, x2, f))
        if k < 256:
            first.append({"trace": trace, "x1": hx(x1), "x2": hx(x2), "f": hx(f),
                          "final_table_sha256": table_sha(sm.table)})
    out.update({"seconds": round(time.time() - t0, 2), "ends": ends,
                "pivot_histogram": {str(k): v for k, v in sorted(hist.items())},
                "total_pivots": sum(k * v for k, v in hist.items()),
                "batch_pivot_sha256": h_p.hexdigest(), "batch_solution_sha256": h_s.hexdigest(),
                "first256": first})
    d["cfg3"] = out
    save_cfg(d)
    print("cfg3:", out["seconds"], "s", ends, out["total_pivots"])


def make_cfg5():
    d = load_cfg()
    for n in (10, 20):
        rows, c = W.klee_minty(n)
        t0 = time.time()
        sm, trace, end, fin = drive(rows.tolist(), c.tolist(), cap=1 << 22)
        d[f"km{n}"] = {
            "generator": {"kind": "klee_minty", "n": n}, "provenance": "reference",
            "end": end, "npiv": len(trace), "first8": trace[:8],
            "pivot_sha256": W.pivot_digest(trace),
            "x1": hx(fin[0]), "x2": hx(fin[1]), "f": hx(fin[2]),
            "final_table_sha256": table_sha(sm.table),
            "final_f_row": [hx(v) for v in sm.table[-1]],
            "final_b": [hx(r[-1]) for r in sm.table[:-1]],
            "row_labels": list(sm.row), "column_labels": list(sm.column),
            "seconds": round(time.time() - t0, 2),
        }
        save_cfg(d)
        print(f"km{n}:", len(trace), "pivots", d[f"km{n}"]["seconds"], "s")


def drive_dantzig(rows, c, cap):
    """The extension rule 'most negative f cell, lowest index on ties' (SURVEY.md §8f N4) driven THROUGH THE
    REFERENCE: outside phase 1 the chosen column is swapped into position 0 of the reference's own table, where its
    first-negative rule (simplex.py:94-98) must take it; pick_element() / recalculate_matrix() then run unmodified
    (ratio scan, arithmetic, label swap) and the columns are swapped back.  Cell arithmetic does not depend on the
    column order, so the result is the reference's own arithmetic under the other entering rule."""
    sm = ref.SimplexMethod([[float(v) for v in r] for r in rows], [float(v) for v in c])
    n, m = sm.n, sm.m
    trace = []

    def swap(j):
        if j == 0:
            return
        for row in sm.table:
            row[0], row[j] = row[j], row[0]
        sm.row[0], sm.row[j] = sm.row[j], sm.row[0]

    try:
        while True:
            phase1 = any(sm.table[i][m] < 0 for i in range(n))
            f = sm.table[n]
            j = 0
            if not phase1:
                best = None
                for q in range(m):
                    if f[q] < 0 and (best is None or f[q] < f[best]):
                        best = q
                j = best if best is not None else 0
            swap(j)
            try:
                ok, i, jj, e = sm.pick_element()
                if not ok:
                    swap(j)
                    return sm, trace, "optimal", (i, jj, e)
                if len(trace) >= cap:
                    swap(j)
                    return sm, trace, "cap", None
                if not phase1:
                    assert jj == 0
                    jj_true = j
                else:
                    jj_true = jj
                trace.append([i, jj_true])
                sm.recalculate_matrix()
            finally:
                pass
            swap(j)
    except ValueError as e:
        swap(j)
        return sm, trace, str(e), None


def make_dantzig():
    """Fixtures of the Dantzig extension rule, produced by the reference itself (see drive_dantzig)."""
    cases = []
    rng = np.random.default_rng(20261019)
    for t in range(150):
        n = int(rng.integers(1, 10))
        m = int(rng.integers(2, 7))
        fam = t % 3
        if fam == 0:
            A = np.round(rng.uniform(-50, 50, (n, m)), 2)
            b = np.round(rng.uniform(-500, 2000, n), 2)
            c = np.round(rng.uniform(-3, 3, m), 2)
        elif fam == 1:
            A = rng.integers(-3, 4, (n, m)).astype(float)
            b = rng.integers(-2, 7, n).astype(float)
            c = rng.integers(-3, 4, m).astype(float)
        else:
            A = -rng.uniform(0.1, 1, (n, m))
            b = rng.uniform(1, 2, n)
            c = -rng.uniform(0.1, 1, m)
        rows = np.hstack([A, b[:, None]]).tolist()
        sm, trace, end, fin = drive_dantzig(rows, c.tolist(), 200)
        cases.append({"name": f"dantzig_{['gui2dp', 'smallint', 'dense'][fam]}_{t:03d}", "provenance": "reference",
                      "rows": [[hx(v) for v in r] for r in rows], "c": [hx(v) for v in c], "cap": 200, "end": end,
                      "trace": trace, "final_table_sha256": table_sha(sm.table),
                      "row_labels": list(sm.row), "column_labels": list(sm.column)})
    for (n, m, seed) in [(30, 40, 1), (64, 33, 2), (17, 96, 3), (40, 700, 4)]:
        rows, c = W.dense_lp(n, m, seed)
        sm, trace, end, fin = drive_dantzig(rows.tolist(), c.tolist(), 400)
        cases.append({"name": f"dantzig_dense_{n}x{m}_seed{seed}", "provenance": "reference",
                      "generator": {"kind": "dense_lp", "n": n, "m": m, "seed": seed}, "cap": 400, "end": end,
                      "trace": trace, "final_table_sha256": table_sha(sm.table),
                      "row_labels": list(sm.row), "column_labels": list(sm.column)})
    with open(os.path.join(HERE, "dantzig_cases.json"), "w") as fh:
        json.dump({"made_by": "tests/golden/make_golden.py dantzig", "rule": "most negative f cell, lowest index on ties "
                   "(extension; entering column only), driven through the reference by a column swap", "cases": cases},
                  fh, indent=0)
    ends = {}
    for cc in cases:
        ends[cc["end"]] = ends.get(cc["end"], 0) + 1
    print("dantzig:", len(cases), "cases", ends)


def make_late():
    """The multi-GPU preflight LP of bench.py (N > 1): tests/util.py::make_lp(96, 4096, 7, "late") — dense_lp with a
    positive objective on the first 95 % of the columns, so the entering column starts on the LAST column block and
    changes owner rank > 100 times on 2 / 4 / 8 ranks.  Provenance "oracle" (549 pivots of a 96 x 4096 table: ~20 min of
    the pure-Python reference); tests/test_oracle.py pins the oracle to the live reference on this LP family."""
    import oracle
    from simplex_method_solver_b200.parallel import column_block
    n, m, seed = 96, 4096, 7
    rows, c = W.dense_lp(n, m, seed)
    c[: int(0.95 * m)] = np.abs(c[: int(0.95 * m)])
    o = oracle.solve(rows, c, max_pivots=100000)
    body = o.table[: n * (m + 1)].reshape(n, m + 1)
    changes = {}
    for world in (2, 4, 8):
        blocks = [column_block(m, r, world) for r in range(world)]
        own = [next(k for k, (a, w) in enumerate(blocks) if a <= int(cc) < a + w) for _, cc in o.trace]
        changes[str(world)] = sum(1 for a, b in zip(own, own[1:]) if a != b)
    out = {"made_by": "tests/golden/make_golden.py late", "provenance": "oracle",
           "generator": "tests/util.py::make_lp(n, m, seed, 'late')", "n": n, "m": m, "seed": seed,
           "input_sha256": W.input_digest(rows, c), "status": int(o.status), "npiv": int(o.npiv),
           "trace": o.trace.tolist(), "pivot_sha256": W.pivot_digest(o.trace),
           "b_sha256": hashlib.sha256(np.ascontiguousarray(body[:, m]).tobytes()).hexdigest(),
           "f_sha256": hashlib.sha256(o.table[n * (m + 1):].tobytes()).hexdigest(),
           "body_checksum_u64": int(W.body_checksum_numpy(body[:, :m])),
           "owner_changes": changes}
    with open(os.path.join(HERE, "late_lp.json"), "w") as fh:
        json.dump(out, fh)
    print("late:", o.status, o.npiv, changes)


def make_cfg4():
    """16384 x 32768 prefix via the oracle (the reference cannot hold this shape)."""
    import ctypes
    import oracle
    d = load_cfg()
    n, m = 16384, 32768
    rows, c = W.dense_lp(n, m, 0)
    out = {"generator": {"kind": "dense_lp", "n": n, "m": m, "seed": 0},
           "input_sha256": W.input_digest(rows, c), "provenance": "oracle"}
    T = np.concatenate([rows.reshape(-1), c])
    del rows
    N = np.empty_like(T)
    K = int(os.environ.get("CFG4_PIVOTS", "2000"))
    trace = []
    marks = {}
    t0 = time.time()
    for k in range(K):
        st, r, cc, e = oracle.pick(T, n, m)
        assert st == oracle.PIVOT
        if k == 0:
            out["first_pivot_value"] = hx(e)
        trace.append([r, cc])
        oracle.lib().orc_update(oracle._dp(T), oracle._dp(N), n, m, r, cc)
        T, N = N, T
        if (k + 1) in (16, 50, 100, 200, 400, 800, 1600, 2000):
            body = T[: n * (m + 1)].reshape(n, m + 1)
            marks[str(k + 1)] = {
                "pivot_sha256": W.pivot_digest(trace),
                "b_first4": [hx(v) for v in body[:4, m]],
                "f_first4": [hx(v) for v in T[n * (m + 1): n * (m + 1) + 4]],
                "b_sha256": hashlib.sha256(np.ascontiguousarray(body[:, m]).tobytes()).hexdigest(),
                "f_sha256": hashlib.sha256(T[n * (m + 1):].tobytes()).hexdigest(),
            }
            print("cfg4 pivot", k + 1, round(time.time() - t0, 1), "s", flush=True)
    out["trace"] = trace
    out["marks"] = marks
    d["cfg4"] = out
    save_cfg(d)


if __name__ == "__main__":
    what = sys.argv[1:] or ["small"]
    for w in what:
        {"small": make_small, "cfg2": make_cfg2, "cfg3": make_cfg3, "cfg5": make_cfg5,
         "cfg4": make_cfg4, "dantzig": make_dantzig, "late": make_late}[w]()
