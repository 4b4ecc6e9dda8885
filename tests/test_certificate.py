"""Certificates of infeasible and unbounded LPs: spx_certificate_batched / _ragged / _split, DeviceBatch.certificate(),
DeviceRaggedBatch.certificate(), batched.certificate() and SimplexMethod.certificate().

CPU part: the Python statement against the C statement (tests/certificate_oracle.c) on every golden final table and
on degenerate random families; hand cases (-0.0, NaN / Inf, labels out of range, repeated labels, an optimal table);
the certificates against the original data and HiGHS, and the rows and columns the solver stopped on; validation of
every entry and of the Python functions.
GPU part: every output's bits against the C statement on both golden sets through DeviceBatch at every engine and
forced cluster size, SimplexMethod after solve() with each loop, a ragged batch against each LP alone, the empty
batch, split tables above 2^24 cells, and a resolve() that makes LPs unbounded.
"""
import ctypes
import math

import numpy as np
import pytest

import certificate_oracle as CO
import oracle
from simplex_method_solver_b200 import workloads as W
from util import case_inputs, flat_of, fresh_lps

NAN = float("nan")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native.load()


def same_bits(a, b):
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    if a.shape != b.shape:
        return False
    an, bn = np.isnan(a), np.isnan(b)     # NaN payloads are not part of the contract
    return bool((an == bn).all() and (a[~an].view(np.uint64) == b[~bn].view(np.uint64)).all())


def assert_cert(got, want, what=""):
    """got, want: (farkas_row, farkas, farkas_bound, ray_col, ray, ray_slope) of one LP"""
    assert int(got[0]) == int(want[0]) and int(got[3]) == int(want[3]), (what, got[0], want[0], got[3], want[3])
    for k in (1, 2, 4, 5):
        assert same_bits(got[k], np.reshape(want[k], np.shape(got[k]))), (what, k)


def lp_of(cert, k):
    """LP k of a batched Certificate in the statement's order"""
    return (cert.farkas_row[k], cert.farkas[k], cert.farkas_bound[k], cert.ray_col[k], cert.ray[k], cert.ray_slope[k])


def split_lp(cert):
    """SimplexMethod.certificate() in the statement's order"""
    return cert.farkas_row, cert.farkas, cert.farkas_bound, cert.ray_col, cert.ray, cert.ray_slope


def stmt(sol):
    return CO.certificate(sol.table, sol.collab.shape[0], sol.rowlab.shape[0], sol.rowlab, sol.collab)


def random_table(n, m, seed, kind):
    """Degenerate tables: exact zeros of both signs, random labels; kind picks which certificate it may hold."""
    g = np.random.default_rng(seed)
    T = g.choice([-1.0, -0.5, -0.0, 0.0, 0.5, 1.0], size=(n, m + 1), p=[0.2, 0.1, 0.15, 0.15, 0.2, 0.2])
    d = g.choice([-1.0, -0.0, 0.0, 1.0], size=m)
    if kind == "feasible":
        T[:, m] = np.abs(T[:, m])
        T[g.random(n) < 0.3, m] = -0.0
    if kind == "ray":
        T[:, m] = np.abs(T[:, m])
        j = int(g.integers(m))
        T[:, j] = np.abs(T[:, j])
        d[j] = -1.0
    if kind == "farkas":
        i = int(g.integers(n))
        T[i, :m] = -np.abs(T[i, :m])
        T[i, m] = -2.0
    perm = g.permutation(n + m).astype(np.int32)
    return np.concatenate([T.reshape(-1), d]), perm[:m].copy(), perm[m:].copy()


# ------------------------------------------------------------------------------------------------- CPU tests
@pytest.mark.parametrize("golden", ["reference", "dantzig"])
def test_python_statement_matches_c_on_golden(golden, ref_cases, dantzig_cases):
    cases = ref_cases if golden == "reference" else dantzig_cases
    for case in cases:
        rows, c = case_inputs(case)
        sol = oracle.solve(rows, c, max_pivots=case["cap"], rule=golden)
        n, m = rows.shape[0], c.shape[0]
        assert_cert(stmt(sol), CO.py_certificate(sol.table, n, m, sol.rowlab, sol.collab), case["name"])


@pytest.mark.parametrize("seed", range(24))
def test_python_statement_matches_c_degenerate(seed):
    n, m = [(1, 1), (3, 2), (7, 5), (20, 30), (30, 8), (12, 12)][seed % 6]
    kind = ("any", "feasible", "ray", "farkas")[seed % 4]
    T, rl, cl = random_table(n, m, seed, kind)
    got = CO.certificate(T, n, m, rl, cl)
    assert_cert(got, CO.py_certificate(T, n, m, rl, cl), seed)
    if kind == "ray":
        assert got[3] >= 0
    if kind == "farkas":
        assert got[0] >= 0


def test_hand_cases():
    # 2 x 2, rows labelled y1 (row 0) and x2 (row 1), columns x1 and y2
    rl, cl = np.array([0, 3], np.int32), np.array([2, 1], np.int32)
    # row 0: b = -1, cells -0.0 and -2: a Farkas row; u[y1] = 1, u[y2] = 0 - (-2) = 2; column x1 is 0 - (-0.0) = +0.0
    T = np.array([-0.0, -2.0, -1.0,
                  1.0, 1.0, 3.0,
                  -1.0, 1.0])
    r, u, ub, c, d, ds = CO.certificate(T, 2, 2, rl, cl)
    assert r == 0 and same_bits(u, [1.0, 2.0]) and ub == -1.0
    assert c == -1 and np.isnan(d).all() and math.isnan(ds)            # b_0 < 0: no ray
    # b = -0.0 counts as >= 0 for the ray and is no Farkas candidate; column 0 has d = -1 and cells -0.0 (>= 0), 1
    T2 = T.copy()
    T2[2] = -0.0
    r, u, ub, c, d, ds = CO.certificate(T2, 2, 2, rl, cl)
    assert r == -1 and np.isnan(u).all() and math.isnan(ub)
    assert c == 0 and ds == -1.0
    assert same_bits(d, [1.0, 1.0])                 # x1 enters (1.0), x2 basic in row 1: T[1][0] + 0.0 = 1.0
    # -0.0 cell in the ray column gives +0.0
    T3 = T2.copy()
    T3[3] = -0.0
    d = CO.certificate(T3, 2, 2, rl, cl)[4]
    assert same_bits(d, [1.0, 0.0]) and not np.signbit(d[1])
    # NaN or Inf in the row or the column disqualifies it; Inf in b too
    for bad in (NAN, math.inf, -math.inf):
        Tb = T.copy()
        Tb[1] = bad
        assert CO.certificate(Tb, 2, 2, rl, cl)[0] == -1
        Tc = T2.copy()
        Tc[3] = bad
        assert CO.certificate(Tc, 2, 2, rl, cl)[3] == -1
        Td = T.copy()
        Td[2] = bad
        assert CO.certificate(Td, 2, 2, rl, cl)[0] == -1
        Te = T2.copy()
        Te[6] = bad
        assert CO.certificate(Te, 2, 2, rl, cl)[3] == -1
    # labels out of range are skipped, never used as an index; a repeated label keeps the statement's last writer
    r, u, ub, c, d, ds = CO.certificate(T, 2, 2, np.array([-5, 99], np.int32), np.array([7, -1], np.int32))
    assert r == 0 and same_bits(u, [0.0, 0.0])
    r, u, *_ = CO.certificate(T, 2, 2, np.array([2, 2], np.int32), np.array([2, 1], np.int32))
    assert same_bits(u, [2.0, 0.0])                 # row label y1 = 1.0, then column 0 (+0.0), then column 1 (2.0)
    # an optimal table: neither
    To = np.array([1.0, -2.0, 3.0, 0.5, 4.0, 0.0, 2.0, 0.0])
    r, u, ub, c, d, ds = CO.certificate(To, 2, 2, rl, cl)
    assert r == -1 and c == -1 and np.isnan(u).all() and np.isnan(d).all()
    for T_, rl_, cl_ in ((T, rl, cl), (T2, rl, cl), (T3, rl, cl), (To, rl, cl),
                         (T, np.array([-5, 99], np.int32), np.array([7, -1], np.int32)),
                         (T, np.array([2, 2], np.int32), np.array([2, 1], np.int32))):
        assert_cert(CO.certificate(T_, 2, 2, rl_, cl_), CO.py_certificate(T_, 2, 2, rl_, cl_))


def verify(rows, c, cert, tol=1e-9):
    """The certificate against the original data of "minimise c.x subject to b + A x >= 0, x >= 0"."""
    r, u, ub, col, d, ds = cert
    m = c.shape[0]
    A, b = rows[:, :m], rows[:, m]
    if r >= 0:
        assert (u >= 0).all() and b @ u < 0
        assert (A.T @ u <= tol * (np.abs(A).T @ u)).all()
        assert abs(b @ u - ub) <= tol * (np.abs(b) @ u + 1.0)
    if col >= 0:
        assert (d >= 0).all() and c @ d < 0
        assert (A @ d >= -tol * (np.abs(A) @ d)).all()
        assert abs(c @ d - ds) <= tol * (np.abs(c) @ d + 1.0)


def dictionary_holds(rows, c, sol, tol=1e-9):
    """The final table is a dictionary of the data: at random points x, the basic variables equal b + T x_N."""
    n, m = rows.shape[0], c.shape[0]
    body = sol.table[: n * (m + 1)].reshape(n, m + 1)
    for seed in range(3):
        x = np.random.default_rng(seed).uniform(0, 1, m)
        val = np.concatenate([x, rows[:, m] + rows[:, :m] @ x])
        want = body[:, m] + body[:, :m] @ val[sol.rowlab]
        if not (np.abs(val[sol.collab] - want) <= tol * (np.abs(body[:, m]) + np.abs(body[:, :m]) @ np.abs(val[sol.rowlab]) + 1)).all():
            return False
    return True


def _highs_status(rows, c):
    """HiGHS without presolve: its presolve reports some of the degenerate unbounded LPs here as infeasible"""
    from scipy.optimize import linprog
    m = c.shape[0]
    return linprog(c, A_ub=-rows[:, :m], b_ub=rows[:, m], bounds=[(0, None)] * m, method="highs",
                   options={"presolve": False}).status


def _failures():
    """(name, rows, c, rule, cap) of LPs that end in a failure: the golden cases and the seeded random families"""
    import json
    import os
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    for fname, rule in (("reference_cases.json", "reference"), ("dantzig_cases.json", "dantzig")):
        with open(os.path.join(here, fname)) as fh:
            for case in json.load(fh)["cases"]:
                if case["end"] in ("incorrect system", "simplex method does not converge"):
                    yield case["name"], *case_inputs(case), rule, case["cap"]
    for fam in ("gui2dp", "smallint", "dense"):
        for k, (rows, c) in enumerate(fresh_lps(fam)):
            yield f"{fam}-{k}", rows, c, "reference", 10000
    for s in range(12):                               # D(n, m) with one column made a free descent: unbounded
        rows, c = W.dense_lp(10 + s, 8 + s, s)
        rows[:, s % 8] = np.abs(rows[:, s % 8])
        yield f"D-unbounded-{s}", rows, c, "dantzig", 10000


def test_certificates_against_the_original_data_and_highs():
    pytest.importorskip("scipy")
    seen = {oracle.INCORRECT: 0, oracle.NOCONV: 0}
    broken = []
    for name, rows, c, rule, cap in _failures():
        sol = oracle.solve(rows, c, max_pivots=cap, rule=rule)
        if sol.status not in seen:
            continue
        seen[sol.status] += 1
        cert = stmt(sol)
        if dictionary_holds(rows, c, sol):
            verify(rows, c, cert)
        else:
            broken.append(name)
        if sol.status == oracle.INCORRECT:
            # the solver stopped on the first row with b < 0, and that row is the certificate
            st, r, _, _ = oracle.pick(sol.table, rows.shape[0], c.shape[0], rule)
            b = sol.table[c.shape[0]: rows.shape[0] * (c.shape[0] + 1): c.shape[0] + 1]
            assert st == oracle.INCORRECT and cert[0] == int(np.flatnonzero(b < 0)[0]), name
            assert _highs_status(rows, c) == 2, name
        else:
            assert cert[3] >= 0, name                  # a finite NOCONV table always has a ray, under either rule
            if rule == "reference":
                f = sol.table[rows.shape[0] * (c.shape[0] + 1):]
                assert cert[3] == int(np.flatnonzero(f < 0)[0]), name      # the solver's entering column
            assert _highs_status(rows, c) == 3, name
    assert seen[oracle.INCORRECT] >= 53 + 29 and seen[oracle.NOCONV] >= 92 + 27 + 12
    assert broken == ["smallint-46"]            # a phase-1 pivot sequence of the reference's arithmetic


def test_optimal_tables_have_neither(ref_cases):
    for case in ref_cases:
        if case["end"] == "optimal":
            rows, c = case_inputs(case)
            cert = stmt(oracle.solve(rows, c, max_pivots=case["cap"]))
            assert cert[0] == -1 and cert[3] == -1, case["name"]


def _err(L):
    return L.spx_last_error().decode()


def test_batched_validation(lib):
    L = lib
    args = [None] * 6
    assert L.spx_certificate_batched(None, 0, 3, 2, None, None, *args, None) == 0
    assert L.spx_certificate_batched(None, -1, 3, 2, None, None, *args, None) == -2
    assert _err(L) == "spx_certificate_batched: bad arguments (B = -1, n = 3, m = 2)"
    assert L.spx_certificate_batched(None, 1, 3, 0, None, None, *args, None) == -2
    assert L.spx_certificate_batched(8, 1, 3, 2, None, 8, *args, None) == -2
    assert _err(L) == "spx_certificate_batched: null T/rowlab/collab"
    assert L.spx_certificate_batched(8, 1, 3, 2, 8, 8, 8, None, None, None, None, None, None) == -2
    assert _err(L) == "spx_certificate_batched: d_row and d_bound need d_farkas (the workspace of the Farkas half)"
    assert L.spx_certificate_batched(8, 1, 3, 2, 8, 8, None, None, None, None, None, 8, None) == -2
    assert _err(L) == "spx_certificate_batched: d_col and d_slope need d_ray (the workspace of the ray half)"
    assert L.spx_certificate_batched(8, 1, 3, 2, 8, 8, *args, None) == 0        # nothing asked for: nothing done


def test_ragged_validation(lib):
    from simplex_method_solver_b200.batched import ragged_plan
    L = lib
    args = [None] * 8
    assert L.spx_certificate_ragged(8, None, 8, *args, None) == -2
    assert _err(L) == "spx_certificate_ragged: null plan"
    plan = ragged_plan([(3, 2), (40, 40)], [10, 10]).plan.copy()
    bad = plan.copy()
    bad[:4] = 0
    assert L.spx_certificate_ragged(8, bad.ctypes.data, 8, *args, None) == -2
    assert _err(L) == "spx_certificate_ragged: h_plan is not a plan of this library (magic / ABI version mismatch)"
    bad = plan.copy()
    bad[8:16].view("<i8")[0] = 3
    assert L.spx_certificate_ragged(8, bad.ctypes.data, 8, *args, None) == -2
    assert _err(L) == "spx_certificate_ragged: inconsistent plan header (B = 3)"
    assert L.spx_certificate_ragged(8, plan.ctypes.data, None, *args, None) == -2
    assert _err(L) == "spx_certificate_ragged: null d_plan/T/rowlab/collab"
    assert L.spx_certificate_ragged(8, plan.ctypes.data, 8, 8, 8, None, None, 8, None, None, None, None) == -2
    assert _err(L) == "spx_certificate_ragged: d_row and d_bound need d_farkas (the workspace of the Farkas half)"
    empty = ragged_plan(np.zeros((0, 2)), []).plan
    assert L.spx_certificate_ragged(None, empty.ctypes.data, None, *args, None) == 0


def test_split_validation(lib):
    L = lib
    args = [None] * 6
    assert L.spx_certificate_split(8, 8, 3, 20, 16, 8, 8, *args, None) == -2
    assert _err(L) == "spx_certificate_split: bad arguments (n = 3, m = 20, ld = 16)"
    assert L.spx_certificate_split(8, None, 3, 2, 16, 8, 8, *args, None) == -2
    assert _err(L) == "spx_certificate_split: null A/b/rowlab/collab"
    assert L.spx_certificate_split(8, 8, 3, 2, 16, 8, 8, None, None, None, 8, None, None, None) == -2
    assert _err(L) == "spx_certificate_split: d_col and d_slope need d_ray (the workspace of the ray half)"


def test_python_validation(lib):
    from simplex_method_solver_b200 import batched
    with pytest.raises(TypeError, match="takes a BatchResult or a RaggedResult"):
        batched.certificate((1, 2))
    z = np.zeros
    bad = batched.BatchResult(z(2, np.int32), z(2, np.int32), z((2, 2)), z(2), z((2, 7)), z((2, 2), np.int32),
                              z((2, 3), np.int32), None, None)
    with pytest.raises(ValueError, match=r"result.tables must be \[B, n\*\(m\+1\)\+m\] = \[2, 11\]"):
        batched.certificate(bad)
    bad = batched.BatchResult(z(2, np.int32), z(2, np.int32), z((2, 2)), z(2), z((2, 11)), z((2, 2), np.int32),
                              z((3, 3), np.int32), None, None)
    with pytest.raises(ValueError, match="result.rowlab must be"):
        batched.certificate(bad)
    plan = batched.ragged_plan([(3, 2)], [10])
    rr = batched.RaggedResult(z(1, np.int32), z(1, np.int32), z(2), z(1), z(10), z(2, np.int32), z(3, np.int32),
                              None, None, np.array([[3, 2, 10]]), plan.offsets)
    with pytest.raises(ValueError, match="result.tables has 10 entries, the shapes need 11"):
        batched.certificate(rr)


def test_sharded_engine_raises(lib):
    from simplex_method_solver_b200.simplex import SimplexMethod
    sm = SimplexMethod.__new__(SimplexMethod)
    sm._sh = object()                    # what engine="sharded" holds instead of a whole table
    with pytest.raises(NotImplementedError, match=r"certificate\(\) is not available with engine='sharded'"):
        sm.certificate()


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


@pytest.mark.gpu
@pytest.mark.parametrize("golden", ["reference", "dantzig"])
def test_golden_every_engine_and_cluster_size(gpu, lib, golden, ref_cases, dantzig_cases):
    batched, N = gpu
    from simplex_method_solver_b200.batched import DeviceBatch, kernel_for
    cases = ref_cases if golden == "reference" else dantzig_cases
    rule = N.RULES[golden]
    orc, bits_of = {}, {}
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
                if S and engine == "global" and S not in (1, 16):
                    continue
                if S and engine == "global" and S < lib.spx_global_min_cluster_size(n, m):
                    continue
                assert lib.spx_set_option(16, S) == 0
                try:
                    db = DeviceBatch(len(idx), n, m, max_pivots=cap, engine=engine)
                    db.upload(tabs)
                    db.run(rule)
                    res, cert = db.result(), db.certificate()
                finally:
                    lib.spx_set_option(16, 0)
                for q, k in enumerate(idx):
                    if k not in orc:
                        sol = oracle.solve(*case_inputs(cases[k]), max_pivots=cap, rule=golden)
                        orc[k] = (sol.status, stmt(sol))
                    assert res.status[q] == orc[k][0]
                    got = lp_of(cert, q)
                    assert_cert(got, orc[k][1], (engine, S, cases[k]["name"]))
                    assert cert.infeasible[q] == (got[0] >= 0) and cert.unbounded[q] == (got[3] >= 0)
                    b = bits_of.setdefault(k, (got[0], got[3], np.asarray(got[1]).tobytes(), np.asarray(got[4]).tobytes()))
                    assert b == (got[0], got[3], np.asarray(got[1]).tobytes(), np.asarray(got[4]).tobytes())
                runs += 1
    assert runs > len(_groups(cases))
    assert any(o[1][0] >= 0 for o in orc.values()) and any(o[1][3] >= 0 for o in orc.values())


@pytest.mark.gpu
@pytest.mark.parametrize("loop", ["classic", "lookahead", "resident", "fused"])
def test_split_after_solve_every_loop(gpu, ref_cases, loop):
    from simplex_method_solver_b200.simplex import SimplexMethod
    done = 0
    for q, case in enumerate(ref_cases):
        if case["end"] == "cap" or (case["end"] == "optimal" and q % 4):       # every failure, a quarter of the rest
            continue
        rows, c = case_inputs(case)
        sm = SimplexMethod(rows, c, engine="stream")
        sol = sm.solve(max_pivots=case["cap"], chunk=17, lookahead=loop)
        ref = oracle.solve(rows, c, max_pivots=case["cap"])
        assert sol.status == ref.status, case["name"]
        cert = sm.certificate()
        assert_cert(split_lp(cert), stmt(ref), (loop, case["name"]))
        assert cert.infeasible == (ref.status == oracle.INCORRECT)
        assert cert.unbounded == (ref.status == oracle.NOCONV)
        done += 1
    assert done > 60


@pytest.mark.gpu
def test_ragged_against_each_lp_alone_and_empty(gpu):
    batched, N = gpu
    shapes = [(8, 2), (4, 3), (20, 20), (100, 100), (128, 256), (600, 800), (30, 30), (12, 5)]
    lps = [W.phase1_lp(n, m, s) if s % 2 else W.dense_lp(n, m, s) for s, (n, m) in enumerate(shapes)]
    lps[2][0][:, 3] = np.abs(lps[2][0][:, 3])                  # unbounded
    lps[3][0][7, :] = -np.abs(lps[3][0][7, :])                 # infeasible (row 7: b < 0, A <= 0)
    lps[6][0][:, 0] = np.abs(lps[6][0][:, 0])
    caps = [64, 64, 300, 2000, 5000, 20000, 3, 64]
    db = batched.DeviceRaggedBatch(shapes, caps, engine="auto_global")
    assert set(db.kernels) == {"smem", "cluster", "global"}
    db.upload(batched.pack_ragged(lps)[1])
    db.run()
    res, cert = db.result(), db.certificate()
    host = batched.certificate(res)
    assert res.status[2] == N.NOCONV and res.status[3] == N.INCORRECT
    for k, (n, m) in enumerate(shapes):
        one = res.lp(k)
        want = CO.certificate(one.tables[0], n, m, one.rowlab[0], one.collab[0])
        assert_cert(lp_of(cert.lp(k), 0), want, k)
        assert_cert(lp_of(host.lp(k), 0), want, ("host", k))
        assert_cert(lp_of(batched.certificate(one), 0), want, ("alone", k))
        verify(*lps[k], want, tol=1e-8)
    assert cert.unbounded[2] and cert.infeasible[3] and not cert.infeasible[0] and not cert.unbounded[0]
    e = batched.certificate(batched.solve_batched(np.zeros((0, 20 * 21 + 20)), 20, 20))
    assert e.farkas.shape == (0, 20) and e.ray.shape == (0, 20) and e.farkas_row.shape == (0,)
    assert batched.DeviceBatch(0, 20, 30).certificate().ray.shape == (0, 30)
    er = batched.certificate(batched.solve_ragged([]))
    assert er.farkas.shape == (0,) and er.infeasible.shape == (0,)
    assert batched.DeviceRaggedBatch(np.zeros((0, 2))).certificate().ray.shape == (0,)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["infeasible", "unbounded"])
def test_split_table_above_2_pow_24_cells(gpu, kind):
    from simplex_method_solver_b200.simplex import SimplexMethod
    n, m = 9000, 2000
    assert n * (m + 1) + m > 1 << 24
    rows, c = W.dense_lp(n, m, 1)
    if kind == "infeasible":
        rows[[4000, 8999], :] = -np.abs(rows[[4000, 8999], :])     # b < 0 and A <= 0 in rows 4000 and 8999
        rows[3000, 5] = 0.5
        rows[3000, m] = -1.0                                        # a candidate row with one positive cell
    else:
        rows[:, [1500, 1999]] = np.abs(rows[:, [1500, 1999]])      # c < 0 and A >= 0 in columns 1500 and 1999
        rows[7, 1000] = 0.0
        rows[:, 1000] = np.abs(rows[:, 1000])
        rows[8, 1000] = -1e-300                                     # a candidate column with one negative cell
    sm = SimplexMethod(rows, c, engine="stream")
    cert = sm.certificate()                                         # the initial table
    rl, cl = sm._dev.labels_host()
    want = CO.certificate(sm._dev.export_flat(sm._npiv), n, m, rl, cl)
    assert_cert(split_lp(cert), want)
    if kind == "infeasible":
        assert cert.farkas_row == 4000 and cert.ray_col == -1
    else:
        assert cert.ray_col == 1500 and cert.farkas_row == -1
    verify(rows, c, want)


@pytest.mark.gpu
def test_resolve_to_unbounded_yields_a_ray(gpu):
    batched, N = gpu
    B, n, m = 6, 20, 20
    data = np.stack([flat_of(*W.dense_lp(n, m, s)) for s in range(B)])
    for k in range(B):                          # column k % m of A made small and >= 0: bounded while its cost is > 0
        body = data[k, : n * (m + 1)].reshape(n, m + 1)
        body[:, k % m] = 1e-3 * np.abs(body[:, k % m])
        data[k, n * (m + 1) + k % m] = 0.5
    res = batched.solve_batched(data, n, m, max_pivots=5000)
    assert (res.status == N.OPTIMAL).all()
    assert not batched.certificate(res).unbounded.any()
    cost = data[:, n * (m + 1):].copy()
    for k in range(0, B, 2):
        cost[k, k % m] = -0.5                   # now unbounded along x_{k % m}
    new = batched.resolve(res, data, cost=cost, max_pivots=5000)
    cert = batched.certificate(new)
    for k in range(B):
        want = CO.certificate(new.tables[k], n, m, new.rowlab[k], new.collab[k])
        assert_cert(lp_of(cert, k), want, k)
        if k % 2 == 0:
            assert new.status[k] == N.NOCONV and cert.unbounded[k]
            rows = data[k, : n * (m + 1)].reshape(n, m + 1)
            verify(rows, cost[k], want)
        else:
            assert new.status[k] == N.OPTIMAL and not cert.unbounded[k] and not cert.infeasible[k]
