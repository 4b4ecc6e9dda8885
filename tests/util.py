"""Helpers shared by the CPU and GPU test modules."""
import hashlib

import numpy as np

END_TO_STATUS = {"optimal": 0, "incorrect system": -1, "simplex method does not converge": -2, "cap": -3}


def unhex(rows):
    return np.asarray([[float.fromhex(v) for v in r] for r in rows], dtype=np.float64)


def unhex1(vals):
    return np.asarray([float.fromhex(v) for v in vals], dtype=np.float64)


def case_inputs(case):
    """rows [n, m+1], c [m] of a golden case (stored as hex floats or as a generator spec)."""
    if "generator" in case:
        from simplex_method_solver_b200 import workloads as W
        g = case["generator"]
        assert g["kind"] == "dense_lp"
        return W.dense_lp(g["n"], g["m"], g["seed"])
    return unhex(case["rows"]), unhex1(case["c"])


def table_sha(flat) -> str:
    return hashlib.sha256(np.ascontiguousarray(flat, dtype="<f8").tobytes()).hexdigest()


def flat_of(rows, c):
    return np.concatenate([np.asarray(rows, dtype=np.float64).reshape(-1), np.asarray(c, dtype=np.float64)])


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def label_codes(names, m):
    """['x1','y2',...] -> int codes used on the device (x_j -> j-1, y_i -> m+i-1)."""
    return [int(s[1:]) - 1 if s[0] == "x" else m + int(s[1:]) - 1 for s in names]


def make_lp(n, m, seed, kind):
    """Test LPs of the sharded flows: rows [n, m+1], c [m].
    dense    : workloads.dense_lp — b > 0, the entering column stays among the FIRST columns (rank 0 owns it)
    late     : dense_lp with a positive objective on the first 95 % of the columns — the entering column starts
               on the LAST column block and then moves between blocks (owner rank != 0, owner changes)
    smallint : small integers — degenerate ties, phase-1 pivots (b < 0), 'incorrect' / 'does not converge' endings
    """
    from simplex_method_solver_b200 import workloads as W
    if kind == "dense":
        return W.dense_lp(n, m, seed)
    if kind == "late":
        rows, c = W.dense_lp(n, m, seed)
        c[: int(0.95 * m)] = np.abs(c[: int(0.95 * m)])
        return rows, c
    assert kind == "smallint", kind
    rng = np.random.default_rng(seed)
    A = rng.integers(-3, 4, (n, m)).astype(float)
    b = rng.integers(-2, 7, n).astype(float)
    c = rng.integers(-3, 4, m).astype(float)
    return np.hstack([A, b[:, None]]), c


def drive_reference(ref, rows, c, cap):
    """Drive the original project's SimplexMethod the way its simplex.py:261-269 does (no Info accumulation).
    Returns (end, trace, final reference-flat table, row labels, column labels)."""
    sm = ref.SimplexMethod([list(map(float, r)) for r in rows], [float(v) for v in c])
    trace = []
    end = "cap"
    while len(trace) < cap:
        try:
            ok, i, j, _e = sm.pick_element()
        except ValueError as e:
            end = str(e)
            break
        if not ok:
            end = "optimal"
            break
        trace.append([i, j])
        sm.recalculate_matrix()
    else:
        # cap reached: is the next pick terminal?  (the oracle reports CAP only on a real pivot)
        try:
            ok, *_ = sm.pick_element()
            end = "cap" if ok else "optimal"
        except ValueError as e:
            end = str(e)
    flat = np.asarray([v for row in sm.table for v in row], dtype=np.float64)
    return end, trace, flat, sm.row, sm.column


FRESH_SHARDED_LPS =[(24, 200, 40, "late"), (40, 400, 64, "late"), (20, 160, 30, "late"), (12, 300, 30, "smallint")]


def fresh_lps(family):
    """The 150 seeded LPs (rows, c) of tests/test_oracle.py::test_oracle_equals_live_reference for one family."""
    rng = np.random.default_rng({"gui2dp": 11, "smallint": 12, "dense": 13}[family])
    for _ in range(150):
        n, m = int(rng.integers(1, 10)), int(rng.integers(2, 7))
        if family == "gui2dp":
            A = np.round(rng.uniform(-50, 50, (n, m)), 2)
            b = np.round(rng.uniform(-500, 2000, n), 2)
            c = np.round(rng.uniform(-3, 3, m), 2)
        elif family == "smallint":
            A = rng.integers(-3, 4, (n, m)).astype(float)
            b = rng.integers(-2, 7, n).astype(float)
            c = rng.integers(-3, 4, m).astype(float)
        else:
            A = -rng.uniform(0.1, 1.0, (n, m)); b = rng.uniform(1.0, 2.0, n); c = -rng.uniform(0.1, 1.0, m)
        yield np.hstack([A, b[:, None]]), c


def fresh_dantzig_lps():
    """The 90 seeded LPs (rows, c) of tests/test_oracle.py::test_dantzig_rule_equals_reference_driven_by_column_swap."""
    rng = np.random.default_rng(77)
    for t in range(90):
        n, m = int(rng.integers(1, 12)), int(rng.integers(2, 9))
        if t % 3 == 0:
            A, b, c = (np.round(rng.uniform(-50, 50, (n, m)), 2), np.round(rng.uniform(-500, 2000, n), 2),
                       np.round(rng.uniform(-3, 3, m), 2))
        elif t % 3 == 1:
            A, b, c = (rng.integers(-3, 4, (n, m)).astype(float), rng.integers(-2, 7, n).astype(float),
                       rng.integers(-3, 4, m).astype(float))
        else:
            A, b, c = -rng.uniform(0.1, 1, (n, m)), rng.uniform(1, 2, n), -rng.uniform(0.1, 1, m)
        yield np.hstack([A, b[:, None]]), c


def owners_of(trace, blocks):
    """owner rank of every pivot's entering column; blocks = [(col0, m_loc), ...]"""
    return [[k for k, (a, w) in enumerate(blocks) if a <= int(cc) < a + w][0] for _, cc in trace]
