"""Sensitivity report of optimal final tables: spx_sensitivity_batched / _ragged / _split, DeviceBatch.sensitivity(),
DeviceRaggedBatch.sensitivity(), batched.sensitivity() and SimplexMethod.sensitivity().

CPU part: an independent pure-Python statement against the sequential C statement (tests/sensitivity_oracle.c) on the
optimal golden cases, degenerate cases and hand cases with empty minima; duals and reduced costs against HiGHS;
perturbations by half and by 1.5 times each finite range; argument validation and error texts (no device).
GPU part: every output's bits against the C statement on both golden sets through DeviceBatch at every engine and
forced cluster size, a mixed K4/K7/K8 ragged batch, host results, SimplexMethod after solve(), get_solution() and
step-API pivots; NaN for LPs that are not optimal; batch independence; the empty batch; a table above 2^24 cells.
"""
import ctypes
import math

import numpy as np
import pytest

import oracle
import sensitivity_oracle as SO
from simplex_method_solver_b200 import workloads as W
from util import case_inputs, flat_of

FIELDS = ("dual", "slack", "reduced_cost", "rhs_range", "cost_range")
INF = math.inf


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native.load()


# ------------------------------------------------------------------------------------------- the statements
def py_sensitivity(T, n, m, rowlab, collab, optimal):
    """The report's tables written out again in plain Python floats, independently of the C statement."""
    nan = float("nan")
    dual, slack, rc = [nan] * n, [nan] * n, [nan] * m
    rr, cr = [[nan, nan] for _ in range(n)], [[nan, nan] for _ in range(m)]
    if not optimal:
        return dual, slack, rc, rr, cr
    T = [float(v) for v in T]
    w = m + 1
    cell = lambda i, j: T[i * w + j]  # noqa: E731
    b = [T[i * w + m] for i in range(n)]
    d = T[n * w:]
    plus0 = lambda v: 0.0 if v == 0 else v  # noqa: E731

    def least(vals):
        best = INF
        for v in vals:
            if v < best:              # NaN never wins
                best = v
        return plus0(best)

    for i in range(n):
        lab = int(collab[i])
        if lab >= m:
            k = lab - m
            dual[k], slack[k], rr[k] = 0.0, plus0(b[i]), [plus0(b[i]), INF]
        else:
            rc[lab] = 0.0
            cr[lab] = [least(d[j] / cell(i, j) for j in range(m) if cell(i, j) > 0),
                       least(d[j] / -cell(i, j) for j in range(m) if cell(i, j) < 0)]
    for j in range(m):
        lab = int(rowlab[j])
        if lab >= m:
            k = lab - m
            dual[k], slack[k] = plus0(-d[j]), 0.0
            rr[k] = [least(b[i] / -cell(i, j) for i in range(n) if cell(i, j) < 0),
                     least(b[i] / cell(i, j) for i in range(n) if cell(i, j) > 0)]
        else:
            rc[lab], cr[lab] = plus0(d[j]), [plus0(d[j]), INF]
    return dual, slack, rc, rr, cr


def same_bits(a, b):
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    if a.shape != b.shape:
        return False
    an, bn = np.isnan(a), np.isnan(b)     # NaN payloads are not part of the contract
    return bool((an == bn).all() and (a[~an].view(np.uint64) == b[~bn].view(np.uint64)).all())


def assert_report(got, want, what=""):
    for name, g, w in zip(FIELDS, got, want):
        assert same_bits(g, np.asarray(w, dtype=np.float64).reshape(np.shape(g))), (what, name)


def oracle_report(sol):
    return SO.sensitivity(sol.table, sol.collab.shape[0], sol.rowlab.shape[0], sol.rowlab, sol.collab,
                          sol.status == oracle.OPTIMAL)


def synthetic(n, m, seed, zeros=0.2):
    """An optimal table (b >= 0, d >= 0) with random labels: columns and rows of both kinds, exact zeros in T, b, d."""
    g = np.random.default_rng(seed)
    T = g.uniform(-1, 1, (n, m + 1))
    T[g.random((n, m + 1)) < zeros] = 0.0
    T[:, m] = np.abs(T[:, m])
    T[g.random(n) < zeros, m] = -0.0
    d = g.uniform(0, 2, m)
    d[g.random(m) < zeros] = 0.0
    perm = g.permutation(n + m).astype(np.int32)
    return np.concatenate([T.reshape(-1), d]), perm[:m].copy(), perm[m:].copy()


# ------------------------------------------------------------------------------------------------- CPU tests
def test_python_statement_matches_c_on_golden(ref_cases):
    seen = 0
    for case in ref_cases:
        if case["end"] != "optimal":
            continue
        rows, c = case_inputs(case)
        sol = oracle.solve(rows, c, max_pivots=case["cap"])
        n, m = rows.shape[0], c.shape[0]
        assert_report(oracle_report(sol), py_sensitivity(sol.table, n, m, sol.rowlab, sol.collab, True), case["name"])
        seen += 1
    assert seen > 100


@pytest.mark.parametrize("seed", range(12))
def test_python_statement_matches_c_degenerate(seed):
    n, m = [(1, 1), (3, 2), (7, 5), (20, 30), (30, 8), (12, 12)][seed % 6]
    T, rl, cl = synthetic(n, m, seed, zeros=0.4)
    assert_report(SO.sensitivity(T, n, m, rl, cl, True), py_sensitivity(T, n, m, rl, cl, True), seed)


def test_hand_cases_empty_minima():
    # 2 x 2, x1 and x2 basic in rows 0 and 1, y1 and y2 nonbasic; T has one sign per column / row so half the
    # minima are over empty sets; b_1 = 0 and d_2 = 0 are degenerate
    T = np.array([1.0, 2.0, 3.0,
                  0.5, 4.0, 0.0,
                  2.0, 0.0])
    rl = np.array([2, 3], np.int32)         # y1, y2 over the columns
    cl = np.array([0, 1], np.int32)         # x1, x2 over the rows
    dual, slack, rc, rr, cr = SO.sensitivity(T, 2, 2, rl, cl, True)
    assert same_bits(dual, [-2.0, 0.0]) and np.signbit(dual[1]) == 0
    assert same_bits(slack, [0.0, 0.0]) and same_bits(rc, [0.0, 0.0])
    assert same_bits(rr, [[INF, 0.0], [INF, 0.0]])      # both columns positive in both rows; b_1 = 0 wins both
    assert same_bits(cr, [[0.0, INF], [0.0, INF]])
    assert_report((dual, slack, rc, rr, cr), py_sensitivity(T, 2, 2, rl, cl, True))
    # not optimal: all NaN, whatever the labels
    for a in SO.sensitivity(T, 2, 2, rl, cl, False):
        assert np.isnan(a).all()


def _highs(rows, c):
    from scipy.optimize import linprog
    m = c.shape[0]
    res = linprog(c, A_ub=-rows[:, :m], b_ub=rows[:, m], bounds=[(0, None)] * m, method="highs")
    assert res.status == 0
    return res


@pytest.mark.parametrize("fam,n,m,seed", [("dense", 10, 10, 1), ("dense", 40, 40, 2), ("dense", 60, 60, 3),
                                          ("dense", 30, 50, 4), ("dense", 50, 20, 5), ("phase1", 20, 20, 6),
                                          ("phase1", 40, 40, 7), ("phase1", 60, 60, 8)])
def test_duals_and_reduced_costs_against_highs(fam, n, m, seed):
    pytest.importorskip("scipy")
    rows, c = (W.dense_lp if fam == "dense" else W.phase1_lp)(n, m, seed)
    sol = oracle.solve(rows, c, max_pivots=100000, rule="dantzig")
    assert sol.status == oracle.OPTIMAL
    dual, slack, rc, rr, cr = oracle_report(sol)
    res = _highs(rows, c)
    scale = lambda a: 1e-9 * np.maximum(1.0, np.abs(a))  # noqa: E731
    assert (np.abs(dual - res.ineqlin.marginals) <= scale(res.ineqlin.marginals)).all()
    assert (np.abs(rc - res.lower.marginals) <= scale(res.lower.marginals)).all()
    assert (np.abs(slack - res.ineqlin.residual) <= 1e-9 * np.maximum(1.0, np.abs(res.ineqlin.residual))).all()


def _resolve(rows, c):
    return oracle.solve(rows, c, max_pivots=100000, rule="dantzig")


def _basis(sol):
    return frozenset(int(v) for v in sol.collab)


@pytest.mark.parametrize("n,m,seed", [(8, 6, 11), (12, 10, 12), (10, 14, 13)])
def test_perturbation_by_half_and_by_one_and_a_half_ranges(n, m, seed):
    rows, c = W.dense_lp(n, m, seed)
    base = _resolve(rows, c)
    assert base.status == oracle.OPTIMAL
    dual, slack, rc, rr, cr = oracle_report(base)
    assert (rr[:, 0] > 0).all() and np.all(np.asarray(base.table[m: n * (m + 1): m + 1]) > 0)   # non-degenerate
    moves = 0
    close = lambda a, b: abs(a - b) <= 1e-8 * max(1.0, abs(b))  # noqa: E731
    for k in range(n):
        for side, sign in ((0, -1.0), (1, 1.0)):
            rng = rr[k, side]
            if not math.isfinite(rng):
                continue
            r2 = rows.copy()
            r2[k, m] += sign * 0.5 * rng
            half = _resolve(r2, c)
            assert half.status == oracle.OPTIMAL and close(half.objm, base.objm + dual[k] * sign * 0.5 * rng), ("b", k, side)
            r2 = rows.copy()
            r2[k, m] += sign * 1.5 * rng
            far = _resolve(r2, c)
            assert far.status != oracle.OPTIMAL or _basis(far) != _basis(base), ("b", k, side)
            moves += 2
    for k in range(m):
        for side, sign in ((0, -1.0), (1, 1.0)):
            rng = cr[k, side]
            if not math.isfinite(rng):
                continue
            c2 = c.copy()
            c2[k] += sign * 0.5 * rng
            half = _resolve(rows, c2)
            assert half.status == oracle.OPTIMAL and close(half.objm, base.objm + sign * 0.5 * rng * base.x[k]), ("c", k)
            c2 = c.copy()
            c2[k] += sign * 1.5 * rng
            far = _resolve(rows, c2)
            assert far.status != oracle.OPTIMAL or _basis(far) != _basis(base), ("c", k, side)
            moves += 2
    assert moves >= n + m


def _err(L):
    return L.spx_last_error().decode()


def test_batched_validation(lib):
    L = lib
    assert L.spx_sensitivity_batched(None, 0, 3, 2, None, None, None, None, None, None, None, None, None) == 0
    assert L.spx_sensitivity_batched(None, -1, 3, 2, None, None, None, None, None, None, None, None, None) == -2
    assert _err(L) == "spx_sensitivity_batched: bad arguments (B = -1, n = 3, m = 2)"
    assert L.spx_sensitivity_batched(None, 1, 0, 2, None, None, None, None, None, None, None, None, None) == -2
    assert L.spx_sensitivity_batched(8, 1, 3, 2, 8, None, 8, None, None, None, None, None, None) == -2
    assert _err(L) == "spx_sensitivity_batched: null T/status/rowlab/collab"


def test_ragged_validation(lib):
    from simplex_method_solver_b200.batched import ragged_plan
    L = lib
    args = [None] * 9
    assert L.spx_sensitivity_ragged(8, None, 8, *args) == -2
    assert _err(L) == "spx_sensitivity_ragged: null plan"
    plan = ragged_plan([(3, 2), (40, 40)], [10, 10]).plan.copy()
    bad = plan.copy()
    bad[:4] = 0
    assert L.spx_sensitivity_ragged(8, bad.ctypes.data, 8, *args) == -2
    assert _err(L) == "spx_sensitivity_ragged: h_plan is not a plan of this library (magic / ABI version mismatch)"
    bad = plan.copy()
    bad[8:16].view("<i8")[0] = 3                       # B no longer matches the launches
    assert L.spx_sensitivity_ragged(8, bad.ctypes.data, 8, *args) == -2
    assert _err(L) == "spx_sensitivity_ragged: inconsistent plan header (B = 3)"
    assert L.spx_sensitivity_ragged(8, plan.ctypes.data, None, *args) == -2
    assert _err(L) == "spx_sensitivity_ragged: null d_plan/T/status/rowlab/collab"
    empty = ragged_plan(np.zeros((0, 2)), []).plan
    assert L.spx_sensitivity_ragged(None, empty.ctypes.data, None, *args) == 0


def test_split_validation(lib):
    L = lib
    opt = ctypes.c_int32(7)
    assert L.spx_sensitivity_split(8, 8, 3, 20, 16, 8, 8, None, None, None, None, None, ctypes.byref(opt), None) == -2
    assert _err(L) == "spx_sensitivity_split: bad arguments (n = 3, m = 20, ld = 16)"
    assert L.spx_sensitivity_split(8, 8, 3, 2, 16, 8, 8, None, None, None, None, None, None, None) == -2
    assert _err(L) == "spx_sensitivity_split: null A/b/rowlab/collab/optimal"
    assert opt.value == 7


def test_python_validation(lib):
    from simplex_method_solver_b200 import batched
    with pytest.raises(TypeError, match="takes a BatchResult or a RaggedResult"):
        batched.sensitivity((1, 2))
    z = np.zeros
    bad = batched.BatchResult(z(2, np.int32), z(2, np.int32), z((2, 2)), z(2), z((2, 7)), z((2, 2), np.int32),
                              z((2, 3), np.int32), None, None)
    with pytest.raises(ValueError, match=r"result.tables must be \[B, n\*\(m\+1\)\+m\] = \[2, 11\]"):
        batched.sensitivity(bad)
    bad = batched.BatchResult(z(2, np.int32), z(2, np.int32), z((2, 2)), z(2), z((2, 11)), z((2, 2), np.int32),
                              z((3, 3), np.int32), None, None)
    with pytest.raises(ValueError, match="result.rowlab must be"):
        batched.sensitivity(bad)


def test_sharded_engine_raises(lib):
    from simplex_method_solver_b200.simplex import SimplexMethod
    sm = SimplexMethod.__new__(SimplexMethod)
    sm._sh = object()                    # what engine="sharded" holds instead of a whole table
    with pytest.raises(NotImplementedError, match=r"sensitivity\(\) is not available with engine='sharded'"):
        sm.sensitivity()


# ------------------------------------------------------------------------------------------------- GPU tests
@pytest.fixture(scope="module")
def gpu(lib):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from simplex_method_solver_b200 import batched, _native
    return batched, _native


def _groups(cases):
    out = {}
    for k, case in enumerate(cases):
        rows, c = case_inputs(case)
        out.setdefault((rows.shape[0], c.shape[0], case["cap"]), []).append(k)
    return out


def _check_uniform(rep, res, what):
    n, m = res.collab.shape[1], res.rowlab.shape[1]
    assert (rep.optimal == (res.status == oracle.OPTIMAL)).all()
    for k in range(res.status.shape[0]):
        want = SO.sensitivity(res.tables[k], n, m, res.rowlab[k], res.collab[k], res.status[k] == oracle.OPTIMAL)
        assert_report([getattr(rep, f)[k] for f in FIELDS], want, (what, k))


@pytest.mark.gpu
@pytest.mark.parametrize("golden", ["reference", "dantzig"])
def test_golden_every_engine_and_cluster_size(gpu, lib, golden, ref_cases, dantzig_cases):
    batched, N = gpu
    from simplex_method_solver_b200.batched import DeviceBatch, kernel_for
    cases = ref_cases if golden == "reference" else dantzig_cases
    rule = N.RULES["dantzig" if golden == "dantzig" else "reference"]
    orc = {}
    runs = 0
    for (n, m, cap), idx in _groups(cases).items():
        tabs = np.stack([flat_of(*case_inputs(cases[k])) for k in idx])
        for engine in ("smem", "cluster", "global"):
            try:
                kernel_for(n, m, engine)
            except ValueError:
                continue
            for S in ((0,) if engine == "smem" else (0, 1, 2, 4, 8, 16)):
                if S and engine == "cluster" and S < lib.spx_cluster_size(n, m):
                    continue
                if S and engine == "global" and S < lib.spx_global_min_cluster_size(n, m):
                    continue
                assert lib.spx_set_option(16, S) == 0
                try:
                    db = DeviceBatch(len(idx), n, m, max_pivots=cap, engine=engine)
                    db.upload(tabs)
                    db.run(rule)
                    res, rep = db.result(), db.sensitivity()
                finally:
                    lib.spx_set_option(16, 0)
                for q, k in enumerate(idx):
                    if k not in orc:
                        sol = oracle.solve(*case_inputs(cases[k]), max_pivots=cap, rule=golden)
                        orc[k] = (sol.status, oracle_report(sol))
                    assert res.status[q] == orc[k][0] and rep.optimal[q] == (orc[k][0] == oracle.OPTIMAL)
                    assert_report([getattr(rep, f)[q] for f in FIELDS], orc[k][1], (engine, S, cases[k]["name"]))
                runs += 1
    assert runs > len(_groups(cases))
    assert any(not v for v in (o[0] == oracle.OPTIMAL for o in orc.values()))      # non-optimal LPs were covered


@pytest.mark.gpu
def test_not_optimal_is_nan(gpu, ref_cases):
    batched, N = gpu
    lps = [(case_inputs(c), c["cap"], c["end"]) for c in ref_cases]
    for end in ("cap", "incorrect system", "simplex method does not converge"):
        (rows, c), cap, _ = next(x for x in lps if x[2] == end)
        res = batched.solve_batched(flat_of(rows, c)[None], rows.shape[0], c.shape[0], max_pivots=cap)
        assert res.status[0] != N.OPTIMAL
        rep = batched.sensitivity(res)
        assert not rep.optimal[0]
        for f in FIELDS:
            assert np.isnan(getattr(rep, f)).all(), (end, f)


@pytest.mark.gpu
def test_ragged_mixed_against_each_lp_alone(gpu):
    batched, N = gpu
    shapes = [(8, 2), (4, 3), (20, 20), (100, 100), (128, 256), (600, 800), (64, 12000), (30, 30)]
    lps = [W.phase1_lp(n, m, s) if s % 2 else W.dense_lp(n, m, s) for s, (n, m) in enumerate(shapes)]
    caps = [64, 64, 300, 2000, 5000, 20000, 20000, 3]                   # the last one stops at its cap
    db = batched.DeviceRaggedBatch(shapes, caps, engine="auto_global")
    assert set(db.kernels) == {"smem", "cluster", "global"}
    db.upload(batched.pack_ragged(lps)[1])
    db.run()
    res, rep = db.result(), db.sensitivity()
    host = batched.sensitivity(res)
    assert not rep.optimal[-1] and rep.optimal.sum() >= 5
    assert any(rep.optimal[k] for k, kind in enumerate(db.kernels) if kind == "global")
    for k, (n, m) in enumerate(shapes):
        one = res.lp(k)
        want = SO.sensitivity(one.tables[0], n, m, one.rowlab[0], one.collab[0], one.status[0] == N.OPTIMAL)
        assert_report([getattr(rep.lp(k), f)[0] for f in FIELDS], want, k)
        assert_report([getattr(host.lp(k), f)[0] for f in FIELDS], want, ("host", k))
        alone = batched.sensitivity(one)
        assert_report([getattr(alone, f)[0] for f in FIELDS], want, ("alone", k))


@pytest.mark.gpu
def test_batch_independence_and_empty(gpu):
    batched, N = gpu
    tabs = np.stack([flat_of(*W.phase1_lp(20, 30, s)) for s in range(6)])
    res = batched.solve_batched(tabs, 20, 30, max_pivots=300)
    rep = batched.sensitivity(res)
    _check_uniform(rep, res, "batch")
    for k in (0, 3, 5):
        one = batched.solve_batched(tabs[k: k + 1], 20, 30, max_pivots=300)
        alone = batched.sensitivity(one)
        assert_report([getattr(alone, f)[0] for f in FIELDS], [getattr(rep, f)[k] for f in FIELDS], k)
    empty = batched.solve_batched(np.zeros((0, 20 * 31 + 30)), 20, 30)
    e = batched.sensitivity(empty)
    assert e.dual.shape == (0, 20) and e.cost_range.shape == (0, 30, 2) and e.optimal.shape == (0,)
    db = batched.DeviceBatch(0, 20, 30)
    assert db.sensitivity().rhs_range.shape == (0, 20, 2)
    er = batched.sensitivity(batched.solve_ragged([]))
    assert er.dual.shape == (0,) and er.optimal.shape == (0,)


@pytest.mark.gpu
def test_table_above_2_pow_24_cells(gpu):
    batched, N = gpu
    n, m = 9000, 2000
    assert n * (m + 1) + m > 1 << 24
    T, rl, cl = synthetic(n, m, 99, zeros=0.05)
    res = batched.BatchResult(np.zeros(1, np.int32), np.zeros(1, np.int32), np.zeros((1, m)), np.zeros(1), T[None],
                              rl[None], cl[None], None, None)
    rep = batched.sensitivity(res)
    _check_uniform(rep, res, "2^24")


def _split_check(sm, rep):
    n, m = sm.n, sm.m
    flat = sm._dev.export_flat(sm._npiv)
    rl, cl = sm._dev.labels_host()
    want = SO.sensitivity(flat, n, m, rl, cl, True)
    assert rep.optimal is True
    assert_report([getattr(rep, f) for f in FIELDS], want)


@pytest.mark.gpu
def test_simplex_method_after_solve_large(gpu):
    from simplex_method_solver_b200.simplex import SimplexMethod
    rows, c = W.dense_lp(1000, 2000, 0)
    sm = SimplexMethod(rows, c)
    sol = sm.solve()
    assert sol.status == 0
    _split_check(sm, sm.sensitivity())


@pytest.mark.gpu
@pytest.mark.parametrize("engine,shape", [("warp", (20, 20)), ("cluster", (128, 256)), ("global", (600, 800))])
def test_simplex_method_after_get_solution(gpu, engine, shape):
    from simplex_method_solver_b200.simplex import SimplexMethod, Error
    rows, c = W.phase1_lp(*shape, 5)
    sm = SimplexMethod(rows, c, engine=engine)
    infos = sm.get_solution(snapshots=False)
    assert not isinstance(infos[-1], Error)
    rep = sm.sensitivity()
    _split_check(sm, rep)
    ref = oracle.solve(rows, c, max_pivots=100000)
    assert_report([getattr(rep, f) for f in FIELDS], oracle_report(ref), engine)


@pytest.mark.gpu
def test_simplex_method_step_api_and_not_optimal(gpu):
    from simplex_method_solver_b200.simplex import SimplexMethod
    rows, c = W.phase1_lp(30, 40, 2)
    sm = SimplexMethod(rows, c)
    with pytest.raises(ValueError, match="needs an optimal table"):
        sm.sensitivity()
    while sm.pick_element()[0]:
        sm.recalculate_matrix()
    rep = sm.sensitivity()
    _split_check(sm, rep)
    assert_report([getattr(rep, f) for f in FIELDS], oracle_report(oracle.solve(rows, c)), "step")
    capped = SimplexMethod(rows, c)
    capped.solve(max_pivots=3)
    with pytest.raises(ValueError, match="needs an optimal table"):
        capped.sensitivity()
