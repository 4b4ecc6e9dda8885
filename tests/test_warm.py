"""Warm start of batched LPs: the change of final tables (spx_warm_change_batched / _ragged), the resume of K4, K7 and
K8 from a table and labels (spx_warm_solve_batched / _ragged), DeviceBatch / DeviceRaggedBatch .change() / .resume()
and batched.resolve().

CPU part: an independent pure-Python statement against the sequential C statement (tests/warm_oracle.c) on random
dictionaries; the algebra (the changed final table equals the trace replayed on the changed LP); changed and resumed
LPs against HiGHS; changes by half a sensitivity range take no pivot; argument validation and error texts.
GPU part: a capped solve resumed equals one longer solve bit for bit on both golden sets, both rules, every engine and
forced cluster size, uniform and ragged; change + resume against the C statement + the oracle's own loop; a resume on
another engine; a table above 2^24 cells; batch independence, the empty batch, and the sensitivity report afterwards.
"""
import ctypes
import math

import numpy as np
import pytest

import oracle
import sensitivity_oracle as SO
import warm_oracle as WO
from simplex_method_solver_b200 import workloads as W
from util import case_inputs, flat_of


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native.load()


# ------------------------------------------------------------------------------------------- the statements
def py_change(T, n, m, rowlab, collab, db, dc):
    """The change written out again in plain Python floats, independently of the C statement."""
    T = [float(v) for v in T]
    w = m + 1
    if db is not None:
        newb = []
        for i in range(n):
            v = T[i * w + m]
            lab = int(collab[i])
            if m <= lab < m + n and float(db[lab - m]) != 0:
                v = v + float(db[lab - m])
            for j in range(m):
                h = int(rowlab[j])
                if m <= h < m + n and float(db[h - m]) != 0:
                    v = v - float(db[h - m]) * T[i * w + j]
            newb.append(v)
        for i in range(n):
            T[i * w + m] = newb[i]
    if dc is not None:
        newd = []
        for j in range(m):
            v = T[n * w + j]
            h = int(rowlab[j])
            if 0 <= h < m and float(dc[h]) != 0:
                v = v + float(dc[h])
            for i in range(n):
                lab = int(collab[i])
                if 0 <= lab < m and float(dc[lab]) != 0:
                    v = v + float(dc[lab]) * T[i * w + j]
            newd.append(v)
        T[n * w:] = newd
    return np.array(T)


def same_bits(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def random_dictionary(n, m, seed, special=False):
    g = np.random.default_rng(seed)
    T = g.standard_normal(n * (m + 1) + m)
    T[g.random(T.size) < 0.2] = 0.0
    if special:
        T[g.integers(0, T.size, 3)] = [np.nan, np.inf, -np.inf]
    lab = g.permutation(n + m).astype(np.int32)
    db, dc = g.standard_normal(n), g.standard_normal(m)
    db[g.random(n) < 0.3] = 0.0
    dc[g.random(m) < 0.3] = -0.0
    return T, lab[:m], lab[m:], db, dc


@pytest.mark.parametrize("n,m,seed,special", [(1, 1, 0, False), (1, 7, 1, False), (7, 1, 2, False), (5, 4, 3, True),
                                              (12, 9, 4, False), (30, 20, 5, True), (9, 30, 6, False)])
def test_python_statement_matches_c(n, m, seed, special):
    T, rl, cl, db, dc = random_dictionary(n, m, seed, special)
    for a, b in ((db, dc), (db, None), (None, dc), (np.zeros(n), -np.zeros(m))):
        want = py_change(T, n, m, rl, cl, a, b)
        got = WO.change(T, n, m, rl, cl, a, b)
        assert same_bits(got, want), (n, m, seed, a is None, b is None)
    # zero changes (-0.0 included) are the identity, NaN and infinities included
    assert same_bits(WO.change(T, n, m, rl, cl, -np.zeros(n), np.zeros(m)), T)


def _lp(n, m, seed, kind):
    return (W.phase1_lp if kind == "phase1" else W.dense_lp)(n, m, seed)


def _with(rows, c, b=None, cc=None):
    rows = rows.copy()
    if b is not None:
        rows[:, -1] = b
    return rows, (c if cc is None else cc)


@pytest.mark.parametrize("n,m,seed,kind", [(8, 6, 1, "dense"), (12, 10, 2, "phase1"), (20, 30, 3, "dense"),
                                           (30, 20, 4, "phase1")])
def test_changed_table_is_the_trace_replayed_on_the_changed_lp(n, m, seed, kind):
    rows, c = _lp(n, m, seed, kind)
    sol = oracle.solve(rows, c)
    g = np.random.default_rng(seed)
    db, dc = g.standard_normal(n) * 0.3, g.standard_normal(m) * 0.3
    T = flat_of(*_with(rows, c, rows[:, -1] + db, c + dc))
    for r, cc in sol.trace:
        T = oracle.update(T, n, m, int(r), int(cc))
    got = WO.change(sol.table, n, m, sol.rowlab, sol.collab, db, dc)
    assert np.allclose(got, T, rtol=1e-9, atol=1e-9 * max(1.0, np.abs(T).max()))


def _highs(rows, c):
    from scipy.optimize import linprog
    A, b = rows[:, :-1], rows[:, -1]
    return linprog(c, A_ub=-A, b_ub=b, bounds=[(0, None)] * c.shape[0], method="highs")


@pytest.mark.parametrize("n,m,seed,kind", [(10, 10, 1, "dense"), (20, 15, 2, "dense"), (12, 10, 3, "phase1"),
                                           (25, 25, 4, "dense")])
def test_change_and_resume_against_highs(n, m, seed, kind):
    rows, c = _lp(n, m, seed, kind)
    sol = oracle.solve(rows, c)
    assert sol.status == oracle.OPTIMAL
    g = np.random.default_rng(100 + seed)
    compared = 0
    for db, dc in ((g.standard_normal(n) * 0.5, None), (None, c * g.uniform(-0.05, 0.05, m)),
                   (g.standard_normal(n), c * g.uniform(-0.2, 0.2, m))):
        b1 = rows[:, -1] + (0 if db is None else db)
        c1 = c + (0 if dc is None else dc)
        T = WO.change(sol.table, n, m, sol.rowlab, sol.collab, db, dc)
        res = WO.resume(T, n, m, sol.rowlab, sol.collab, c1, 100000)
        ref = _highs(*_with(rows, c, b1, c1))
        if res.status != oracle.OPTIMAL:
            continue              # the reference's phase 1 may end elsewhere; only optimal LPs are compared
        assert ref.status == 0
        assert math.isclose(res.objm, ref.fun, rel_tol=1e-8, abs_tol=1e-8)
        assert (res.x >= -1e-9).all() and (b1 + rows[:, :-1] @ res.x >= -1e-7 * (1 + np.abs(b1))).all()
        compared += 1
    assert compared >= 1


def _ranges(sol, n, m):
    return SO.sensitivity(sol.table, n, m, sol.rowlab, sol.collab, True)


@pytest.mark.parametrize("n,m,seed", [(8, 6, 11), (12, 10, 12), (10, 14, 13)])
def test_change_by_half_a_range_takes_no_pivot(n, m, seed):
    rows, c = W.dense_lp(n, m, seed)
    sol = oracle.solve(rows, c)
    assert sol.status == oracle.OPTIMAL
    _, _, _, rr, cr = _ranges(sol, n, m)
    checked = 0
    for k in range(n):
        for side, sign in ((0, -1.0), (1, 1.0)):
            if not math.isfinite(rr[k, side]) or rr[k, side] == 0:
                continue
            db = np.zeros(n)
            db[k] = sign * rr[k, side] / 2
            T = WO.change(sol.table, n, m, sol.rowlab, sol.collab, db, None)
            res = WO.resume(T, n, m, sol.rowlab, sol.collab, c, 1000)
            assert res.status == oracle.OPTIMAL and res.npiv == 0, (k, side)
            w = m + 1
            for i in range(n):
                if sol.collab[i] < m:
                    assert res.x[sol.collab[i]] == T[i * w + m]
            checked += 1
    for k in range(m):
        for side, sign in ((0, -1.0), (1, 1.0)):
            if not math.isfinite(cr[k, side]) or cr[k, side] == 0:
                continue
            dc = np.zeros(m)
            dc[k] = sign * cr[k, side] / 2
            T = WO.change(sol.table, n, m, sol.rowlab, sol.collab, None, dc)
            res = WO.resume(T, n, m, sol.rowlab, sol.collab, c + dc, 1000)
            assert res.status == oracle.OPTIMAL and res.npiv == 0, (k, side)
            checked += 1
    assert checked >= n


def _err(L):
    return L.spx_last_error().decode()


def test_c_entries_validation(lib):
    L = lib
    p = ctypes.c_void_p(16)
    rl = cl = p
    assert L.spx_warm_change_batched(None, 0, 4, 2, None, None, None, None, None) == 0
    assert L.spx_warm_change_batched(p, 3, 4, 2, None, None, None, None, None) == 0       # no delta: nothing to do
    assert L.spx_warm_change_batched(p, -1, 4, 2, rl, cl, p, p, None) == -2
    assert "bad arguments" in _err(L)
    assert L.spx_warm_change_batched(p, 3, 0, 2, rl, cl, p, p, None) == -2
    assert L.spx_warm_change_batched(p, 3, 4, 2, None, cl, p, None, None) == -2
    assert "spx_warm_change_batched: null T/rowlab/collab" in _err(L)
    assert L.spx_warm_change_ragged(None, None, None, None, None, p, p, None) == -2
    assert "spx_warm_change_ragged: null plan" in _err(L)
    junk = (ctypes.c_char * 4096)()
    assert L.spx_warm_change_ragged(None, junk, None, None, None, p, p, None) == -2
    assert "not a plan of this library" in _err(L)
    # uniform solve: engine, shape, pointers, labels, function, rule, capacity
    args = lambda **kw: [kw.get("engine", 1), p, kw.get("B", 2), kw.get("n", 4), kw.get("m", 2), kw.get("rule", 0),  # noqa: E731
                         kw.get("cap", 8), kw.get("fn", p), p, kw.get("obj", p), p, p, kw.get("rl", rl),
                         kw.get("cl", cl), None, None, None]
    assert L.spx_warm_solve_batched(*args(engine=3)) == -2 and "unknown engine 3" in _err(L)
    assert L.spx_warm_solve_batched(*args(cap=-1)) == -2 and "spx_warm_solve_batched: bad arguments" in _err(L)
    assert L.spx_warm_solve_batched(*args(rl=None)) == -2 and "null rowlab/collab" in _err(L)
    assert L.spx_warm_solve_batched(*args(fn=None)) == -2 and "null function with obj" in _err(L)
    assert L.spx_warm_solve_batched(*args(rule=7)) == -2 and "unknown rule 7" in _err(L)
    assert L.spx_warm_solve_batched(*args(engine=1, n=200, m=200)) == -2
    assert _err(L).startswith("spx_warm_solve_batched: ") and "exceed" in _err(L)
    assert L.spx_warm_solve_batched(*args(B=0, rl=None, cl=None, fn=None)) == 0
    assert L.spx_warm_solve_ragged(None, None, None, 0, None, None, None, None, None, None, None, None, None,
                                   None) == -2
    assert "spx_warm_solve_ragged: null plan" in _err(L)


def _plan(shapes, caps, engine="auto"):
    from simplex_method_solver_b200.batched import ragged_plan
    return ragged_plan(shapes, caps, engine)


def test_ragged_validation_and_empty_plan(lib):
    L = lib
    p = ctypes.c_void_p(16)
    plan = _plan(np.zeros((0, 2)), np.zeros(0))
    h = plan.plan.ctypes.data
    assert L.spx_warm_change_ragged(None, h, None, None, None, p, p, None) == 0
    assert L.spx_warm_solve_ragged(None, h, None, 0, None, None, None, None, None, None, None, None, None, None) == 0
    plan = _plan([(4, 2), (20, 20)], [8, 8])
    h = plan.plan.ctypes.data
    assert L.spx_warm_change_ragged(p, h, p, None, p, p, p, None) == -2
    assert "spx_warm_change_ragged: null d_plan/T/rowlab/collab" in _err(L)
    assert L.spx_warm_change_ragged(p, h, p, p, p, None, None, None) == 0
    assert L.spx_warm_solve_ragged(p, h, p, 0, p, p, p, p, p, None, p, None, None, None) == -2
    assert "spx_warm_solve_ragged: null rowlab/collab" in _err(L)
    assert L.spx_warm_solve_ragged(p, h, p, 0, None, p, p, p, p, p, p, None, None, None) == -2
    assert "null function with obj" in _err(L)
    assert L.spx_warm_solve_ragged(p, h, p, 5, p, p, p, p, p, p, p, None, None, None) == -2
    assert "unknown rule 5" in _err(L)


def test_python_validation(lib):
    from simplex_method_solver_b200.batched import BatchResult, RaggedResult, resolve
    rows, c = W.dense_lp(6, 4, 1)
    sol = oracle.solve(rows, c)
    T = np.stack([flat_of(rows, c)] * 3)
    z = np.zeros
    res = BatchResult(z(3, np.int32), z(3, np.int32), z((3, 4)), z(3), np.stack([sol.table] * 3),
                      np.stack([sol.rowlab] * 3), np.stack([sol.collab] * 3), None, None)
    bad = res._replace(rowlab=res.rowlab.copy())
    bad.rowlab[2, 0] = bad.rowlab[2, 1]
    with pytest.raises(ValueError, match="LP 2: labels are not a permutation of 0..9"):
        resolve(bad, T)
    rhs = np.tile(rows[:, -1], (3, 1))
    rhs[1, 3] = np.nan
    with pytest.raises(ValueError, match="LP 1: rhs - old rhs is not finite"):
        resolve(res, T, rhs=rhs)
    cost = np.tile(c, (3, 1))
    cost[0, 0] = np.inf
    with pytest.raises(ValueError, match="LP 0: cost - old cost is not finite"):
        resolve(res, T, cost=cost)
    with pytest.raises(ValueError, match=r"rhs must be \[3, 6\] or \[6\]"):
        resolve(res, T, rhs=np.zeros(5))
    with pytest.raises(ValueError, match="data must be"):
        resolve(res, T[:2])
    rr = RaggedResult(z(2, np.int32), z(2, np.int32), z(8), z(2), np.concatenate([sol.table] * 2),
                      np.concatenate([sol.rowlab] * 2), np.concatenate([sol.collab] * 2), None, None,
                      np.array([[6, 4, 8]] * 2), z((2, 5), np.int64))
    lps = [(rows, c), (rows, c)]
    with pytest.raises(ValueError, match="LP 1: rhs - old rhs is not finite"):
        resolve(rr, lps, rhs=[rows[:, -1], np.full(6, np.nan)])
    badr = rr._replace(collab=rr.collab.copy())
    badr.collab[6] = 99
    with pytest.raises(ValueError, match="LP 1: labels are not a permutation"):
        resolve(badr, lps)
    with pytest.raises(ValueError, match="shapes differ"):
        resolve(rr, [(rows, c)])


# ------------------------------------------------------------------------------------------------ GPU
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


def _engines(lib, n, m):
    from simplex_method_solver_b200.batched import kernel_for
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
            yield engine, S


def _forced(lib, S, fn):
    assert lib.spx_set_option(16, S) == 0
    try:
        return fn()
    finally:
        lib.spx_set_option(16, 0)


def _solve(batched, tabs, n, m, cap, engine, rule, function=None, labels=None):
    """a cold solve (function None) or a resume of tabs with labels, snapshots on"""
    db = batched.DeviceBatch(tabs.shape[0], n, m, max_pivots=cap, snapshots=True, engine=engine)
    db.upload(tabs)
    if function is None:
        db.run(rule)
    else:
        db.upload_labels(*labels)
        db.resume(function, rule)
    return db.result()


def _check_continuation(full, a, b, K, what):
    """full = one solve at cap 2K; a = the solve at cap K, b = its resume at cap K"""
    for q in range(full.status.shape[0]):
        k1, k2 = int(a.npiv[q]), int(b.npiv[q])
        assert int(full.status[q]) == int(b.status[q]), (what, q)
        assert int(full.npiv[q]) == k1 + k2, (what, q)
        if int(a.status[q]) != oracle.CAP:
            assert k2 == 0 and int(b.status[q]) == int(a.status[q]), (what, q)
        tr = np.concatenate([a.trace[q, :k1], b.trace[q, :k2]])
        assert full.trace[q, : k1 + k2].tobytes() == tr.tobytes(), (what, q)
        sn = np.concatenate([a.snaps[q, :k1], b.snaps[q, : k2 + 1]])
        assert full.snaps[q, : k1 + k2 + 1].tobytes() == sn.tobytes(), (what, q)
    for f in ("tables", "rowlab", "collab", "x", "obj"):
        assert getattr(full, f).tobytes() == getattr(b, f).tobytes(), (what, f)


@pytest.mark.gpu
@pytest.mark.parametrize("golden", ["reference", "dantzig"])
def test_continuation_every_engine_and_cluster_size(gpu, lib, golden, ref_cases, dantzig_cases):
    batched, N = gpu
    cases = ref_cases if golden == "reference" else dantzig_cases
    rule = N.RULES[golden]
    runs = 0
    for (n, m, cap), idx in _groups(cases).items():
        tabs = np.stack([flat_of(*case_inputs(cases[k])) for k in idx])
        K = max(1, min(cap, 4000) // 2)
        function = tabs[:, n * (m + 1):]
        for engine, S in _engines(lib, n, m):
            def go():
                full = _solve(batched, tabs, n, m, 2 * K, engine, rule)
                a = _solve(batched, tabs, n, m, K, engine, rule)
                b = _solve(batched, a.tables, n, m, K, engine, rule, function, (a.rowlab, a.collab))
                return full, a, b
            full, a, b = _forced(lib, S, go)
            _check_continuation(full, a, b, K, (golden, n, m, engine, S))
            runs += 1
    assert runs > len(_groups(cases))


@pytest.mark.gpu
def test_continuation_ragged_mixed(gpu):
    batched, N = gpu
    lps, _ = W.mixed_large_lps(96, seed=5)
    K = 24
    shapes, packed = batched.pack_ragged(lps)
    function = np.concatenate([c for _, c in lps])

    def run(cap, tables=None, labels=None):
        db = batched.DeviceRaggedBatch(shapes, cap, snapshots=True, engine="auto_global")
        db.upload(packed if tables is None else tables)
        if labels is None:
            db.run()
        else:
            db.upload_labels(*labels)
            db.resume(function)
        return db.result()
    full = run(2 * K)
    a = run(K)
    b = run(K, a.tables, (a.rowlab, a.collab))
    assert {k for k in ("smem", "cluster", "global")} <= set(batched.kernels_for(shapes, "auto_global"))
    assert (a.status != oracle.CAP).any() and (a.status == oracle.CAP).any()
    for k in range(len(lps)):
        f, x, y = full.lp(k), a.lp(k), b.lp(k)
        _check_continuation(f._replace(trace=f.trace[:, :2 * K], snaps=f.snaps), x, y, K, ("ragged", k))


def _statement(tables, n, m, rowlab, collab, db, dc, function, cap, rule):
    out = []
    for q in range(tables.shape[0]):
        T = WO.change(tables[q], n, m, rowlab[q], collab[q], None if db is None else db[q],
                      None if dc is None else dc[q])
        out.append((T, WO.resume(T, n, m, rowlab[q], collab[q], function[q], cap, rule)))
    return out


def _check_statement(res, want, what):
    for q, (Tchg, o) in enumerate(want):
        assert (int(res.status[q]), int(res.npiv[q])) == (o.status, o.npiv), (what, q)
        assert res.trace[q, : o.npiv].tobytes() == o.trace.tobytes(), (what, q)
        assert res.tables[q].tobytes() == o.table.tobytes(), (what, q)
        assert res.rowlab[q].tobytes() == o.rowlab.tobytes() and res.collab[q].tobytes() == o.collab.tobytes()
        assert res.x[q].tobytes() == o.x.tobytes() and res.obj[q] == o.obj2, (what, q)


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,kind,engine,B", [(6, 4, "dense", "smem", 24), (20, 30, "phase1", "smem", 16),
                                               (128, 256, "phase1", "cluster", 3), (600, 800, "dense", "global", 1)])
def test_change_and_resume_against_statement(gpu, n, m, kind, engine, B):
    batched, N = gpu
    lps = [_lp(n, m, 40 + s, kind) for s in range(B)]
    tabs = np.stack([flat_of(r, c) for r, c in lps])
    base = batched.solve_batched(tabs, n, m, max_pivots=20000, engine=engine)
    b0 = tabs[:, : n * (m + 1)].reshape(B, n, m + 1)[:, :, m]
    c0 = tabs[:, n * (m + 1):]
    g = np.random.default_rng(n + m)
    cases = {"rhs": (b0 + g.standard_normal((B, n)) * np.abs(b0).mean() * 0.5, None),
             "cost": (None, c0 * (1 + g.uniform(-0.05, 0.05, (B, m)))),
             "both": (b0 * g.uniform(0.5, 1.5, (B, n)) - 0.2 * np.abs(b0).mean(), c0 * g.uniform(0.8, 1.2, (B, m))),
             "zero": (b0, c0)}
    statuses = set()
    for name, (rhs, cost) in cases.items():
        res = batched.resolve(base, tabs, rhs=rhs, cost=cost, max_pivots=20000, engine=engine)
        db = None if rhs is None else rhs - b0
        dc = None if cost is None else cost - c0
        _check_statement(res, _statement(base.tables, n, m, base.rowlab, base.collab, db, dc,
                                         c0 if cost is None else cost, 20000, "reference"), (name, engine))
        if name == "zero":
            assert res.tables.tobytes() == base.tables.tobytes() and (res.npiv == 0).all()
        statuses |= set(int(s) for s in res.status)
    assert oracle.OPTIMAL in statuses


@pytest.mark.gpu
def test_change_to_phase1_incorrect_and_nonconvergent(gpu):
    batched, N = gpu
    # x1 + x2 <= 10, 2 x1 <= 8, minimise x1 + x2: optimal at 0 in the first dictionary
    rows = np.array([[-1.0, -1.0, 10.0], [-2.0, 0.0, 8.0], [0.0, -1.0, 6.0]])
    c = np.array([1.0, 1.0])
    tabs = np.stack([flat_of(rows, c)] * 4)
    base = batched.solve_batched(tabs, 3, 2, max_pivots=50)
    rhs = np.array([[10.0, 8.0, 6.0], [-5.0, 8.0, 6.0], [4.0, 8.0, -3.0], [10.0, 8.0, 6.0]])   # -, infeasible x2
    cost = np.array([[1.0, 1.0], [1.0, 1.0], [1.0, 1.0], [-1.0, -1.0]])                       # -, -, -, max x1 + x2
    res = batched.resolve(base, tabs, rhs=rhs, cost=cost, max_pivots=50)
    want = _statement(base.tables, 3, 2, base.rowlab, base.collab, rhs - rows[:, -1], cost - c, cost, 50,
                      "reference")
    _check_statement(res, want, "hand")
    assert int(res.status[1]) == oracle.INCORRECT and int(res.status[2]) == oracle.INCORRECT
    # unbounded: minimise -x2 when only x1 is bounded
    rows2 = np.array([[-1.0, 0.0, 10.0], [-2.0, 0.0, 8.0]])
    t2 = np.stack([flat_of(rows2, c)])
    b2 = batched.solve_batched(t2, 2, 2, max_pivots=50)
    r2 = batched.resolve(b2, t2, cost=np.array([[1.0, -1.0]]), max_pivots=50)
    _check_statement(r2, _statement(b2.tables, 2, 2, b2.rowlab, b2.collab, None, np.array([[0.0, -2.0]]),
                                    np.array([[1.0, -1.0]]), 50, "reference"), "unbounded")
    assert int(r2.status[0]) == oracle.NOCONV


@pytest.mark.gpu
@pytest.mark.parametrize("first,then", [("cluster", "smem"), ("cluster", "global"), ("global", "cluster")])
def test_resume_on_another_engine(gpu, lib, first, then):
    batched, N = gpu
    n, m, B = 20, 30, 12
    tabs = np.stack([flat_of(*W.phase1_lp(n, m, 70 + s)) for s in range(B)])
    K = 6
    function = tabs[:, n * (m + 1):]
    full = _solve(batched, tabs, n, m, 2 * K, first, N.RULE_REFERENCE)
    a = _solve(batched, tabs, n, m, K, first, N.RULE_REFERENCE)
    for S in (0, 2):
        b = _forced(lib, S, lambda: _solve(batched, a.tables, n, m, K, then, N.RULE_REFERENCE, function,
                                           (a.rowlab, a.collab)))
        _check_continuation(full, a, b, K, (first, then, S))


@pytest.mark.gpu
def test_change_table_above_2_pow_24_cells(gpu):
    batched, N = gpu
    import torch
    n, m = 9000, 2000
    assert n * (m + 1) + m > 1 << 24
    g = np.random.default_rng(7)
    T = g.standard_normal(n * (m + 1) + m)
    lab = g.permutation(n + m).astype(np.int32)
    db, dc = g.standard_normal(n), g.standard_normal(m)
    db[g.random(n) < 0.5] = 0.0
    dv = batched.DeviceBatch(1, n, m, max_pivots=0, trace=False, engine="global")
    dv.upload(T[None])
    dv.upload_labels(lab[None, :m], lab[None, m:])
    dv.change(db, dc)
    got = dv.T[0].cpu().numpy()
    assert got.tobytes() == WO.change(T, n, m, lab[:m], lab[m:], db, dc).tobytes()


@pytest.mark.gpu
def test_batch_independence_empty_and_sensitivity(gpu):
    batched, N = gpu
    n, m = 20, 30
    tabs = np.stack([flat_of(*W.phase1_lp(n, m, s)) for s in range(6)])
    base = batched.solve_batched(tabs, n, m, max_pivots=300)
    g = np.random.default_rng(3)
    cost = tabs[:, n * (m + 1):] * g.uniform(0.9, 1.1, (6, m))
    res = batched.resolve(base, tabs, cost=cost, max_pivots=300)
    for k in (0, 3, 5):
        one = batched.resolve(batched.BatchResult(*[None if v is None else v[k: k + 1] for v in base]),
                              tabs[k: k + 1], cost=cost[k: k + 1], max_pivots=300)
        for f in ("status", "npiv", "tables", "x", "obj", "rowlab", "collab"):
            assert getattr(one, f)[0].tobytes() == getattr(res, f)[k].tobytes(), (k, f)
    rep = batched.sensitivity(res)
    for k in range(6):
        want = SO.sensitivity(res.tables[k], n, m, res.rowlab[k], res.collab[k], res.status[k] == oracle.OPTIMAL)
        for g_, w in zip([rep.dual[k], rep.slack[k], rep.reduced_cost[k], rep.rhs_range[k], rep.cost_range[k]], want):
            g_, w = np.asarray(g_), np.asarray(w).reshape(np.shape(g_))
            assert (np.isnan(g_) == np.isnan(w)).all() and g_[~np.isnan(g_)].tobytes() == w[~np.isnan(w)].tobytes()
    e = batched.resolve(batched.solve_batched(np.zeros((0, n * (m + 1) + m)), n, m), np.zeros((0, n * (m + 1) + m)))
    assert e.status.shape == (0,) and e.tables.shape == (0, n * (m + 1) + m)
    er = batched.resolve(batched.solve_ragged([]), [])
    assert er.status.shape == (0,)
    dv = batched.DeviceBatch(0, n, m)
    dv.change(np.zeros(n), np.zeros(m))
    dv.resume(np.zeros(m))
