"""Dantzig's rule with Bland's rule on degenerate pivots and a ratio-tested phase 1 (SPX_RULE_DANTZIG_BLAND): its
statements and the batched engines that run it.

CPU part: an independent pure-Python statement (dantzig_bland_model.py) equals the sequential C statement
(dantzig_bland_oracle.c) bit for bit on the golden cases, seeded dense, phase-1 and scaled families, Klee-Minty and
non-finite tables; the statement ends every finite golden case in a terminal status that HiGHS confirms, ends the
reference's cycling example and the 1000 x 1000 phase-1 LP that caps under every other rule, and never makes a
feasible row infeasible; the C ABI and SimplexMethod refuse the rule outside the batched entries.
GPU part: K4 (warp and CTA mode), K7 at every cluster size and K8 at every S under the rule, uniform and ragged, at the
capacity edges and on non-finite inputs, capped-and-resumed solves and re-solves, bit for bit against the statement;
the certificates of the LPs it stops on.
"""
import re

import numpy as np
import pytest

import dantzig_bland_model as M
import dantzig_bland_oracle as D
import oracle
from simplex_method_solver_b200 import workloads as W
from test_capacity_edges import (EDGES, SIZES, SPECIAL_CAP, SPECIAL_RUNS, SPECIAL_SHAPES, _cap, edge_batch,
                                 engine_runs, same, special_lps)
from test_cluster_batched import cluster_size
from test_devex import FAKE, UNIFORM, _refused, families, nonfinite_tables, scaled, uniform_batch
from util import case_inputs, flat_of

HEADER_RULE = re.compile(r"#define SPX_RULE_DANTZIG_BLAND\s+(\d+)")
RULE = "dantzig_bland"


def model_equals_oracle(T, n, m, cap, what, rowlab=None, collab=None):
    o = D.solve_flat(T, n, m, cap, rowlab=rowlab, collab=collab)
    st, trace, table, rl, cl = M.solve(T, n, m, cap, rowlab, collab)
    assert (st, len(trace)) == (o.status, o.npiv), what
    assert [tuple(t) for t in o.trace.tolist()] == trace, what
    assert same(np.asarray(table), o.table), what
    assert rl == o.rowlab.tolist() and cl == o.collab.tolist(), what
    return o


def hand_tables():
    """(name, n, m, flat, rowlab, collab) of tables whose ratios are -0.0, NaN and +inf, with shuffled labels"""
    nan, inf = float("nan"), float("inf")
    out = []
    # phase 2, column 0 enters: row 0 has b = -0.0 (a -0 ratio, degenerate), row 1 b = NaN (a NaN ratio)
    out.append(("-0 and NaN ratios", 3, 2, np.array([-1.0, 1.0, -0.0, -2.0, 1.0, nan, -1.0, -1.0, 4.0,
                                                     -3.0, -1.0]), [3, 1], [0, 4, 2]))
    # phase 1 with +inf in the target row and a NaN cell elsewhere
    out.append(("inf target", 3, 3, np.array([inf, 1.0, 2.0, -1.0, -1.0, nan, 0.0, 2.0, -2.0, -1.0, 3.0, 1.0,
                                              -1.0, -2.0, 0.5]), None, None))
    # ties on every key: equal ratios, equal scores
    out.append(("ties", 4, 2, np.array([-1.0, -1.0, 1.0, -1.0, -1.0, 1.0, -2.0, -2.0, 2.0, 1.0, 1.0, 0.0,
                                        -1.0, -1.0]), [5, 2], [0, 4, 1, 3]))
    return out


# --------------------------------------------------------------------------- CPU: the rule
def test_model_equals_oracle_on_the_golden_cases(ref_cases):
    assert len(ref_cases) == 381
    for case in ref_cases:
        rows, c = case_inputs(case)
        rows = np.asarray(rows, dtype=np.float64)
        model_equals_oracle(flat_of(rows, c), rows.shape[0], rows.shape[1] - 1, 300, case.get("name", case))


def test_model_equals_oracle_on_seeded_scaled_and_non_finite_tables():
    ends = set()
    for name, rows, c in families():
        o = model_equals_oracle(flat_of(rows, c), rows.shape[0], rows.shape[1] - 1, 2000, name)
        ends.add(o.status)
    assert oracle.OPTIMAL in ends
    for name, n, m, T in nonfinite_tables():
        model_equals_oracle(T, n, m, 40, name)
    for name, n, m, T, rl, cl in hand_tables():
        rl = None if rl is None else np.array(rl, np.int32)
        cl = None if cl is None else np.array(cl, np.int32)
        model_equals_oracle(T, n, m, 40, name, rl, cl)


def test_degenerate_step_takes_blands_column():
    # phase 2: Dantzig's column 1 (f = -3) has a zero ratio (row 0, b = 0); Bland's column is the lowest header label
    T = np.array([1.0, -1.0, 0.0,
                  -1.0, -1.0, 4.0,
                  -1.0, -3.0])
    assert D.pick(T, 2, 2) == (oracle.PIVOT, 1, 0)
    assert D.pick(T, 2, 2, rowlab=np.array([7, 2], np.int32), collab=np.array([0, 1], np.int32)) == (oracle.PIVOT, 0, 1)


def _highs(rows, c):
    from scipy.optimize import linprog
    m = c.shape[0]
    res = linprog(c, A_ub=-rows[:, :m], b_ub=rows[:, m], bounds=[(0, None)] * m, method="highs")
    if res.status == 2:
        # HiGHS may call an unbounded LP infeasible: a zero-cost solve tells whether a feasible point exists
        feas = linprog(np.zeros(m), A_ub=-rows[:, :m], b_ub=rows[:, m], bounds=[(0, None)] * m, method="highs")
        if feas.status == 0:
            return 3, None
    return res.status, res.fun


def test_every_finite_golden_case_ends_as_highs_says(ref_cases):
    pytest.importorskip("scipy")
    code = {oracle.OPTIMAL: 0, oracle.INCORRECT: 2, oracle.NOCONV: 3}
    seen = 0
    for case in ref_cases:
        rows, c = case_inputs(case)
        rows = np.asarray(rows, dtype=np.float64)
        if not (np.isfinite(rows).all() and np.isfinite(c).all()):
            continue
        seen += 1
        n, m = rows.shape[0], c.shape[0]
        o = D.solve_flat(flat_of(rows, c), n, m, 2000)
        assert o.status in code, case["name"]
        st, fun = _highs(rows, c)
        assert code[o.status] == st, case["name"]
        if st == 0:
            assert abs(o.objm - fun) <= 1e-7 * max(1.0, abs(fun)), case["name"]
    assert seen == 381


def test_the_references_cycling_example_ends_unbounded(ref_cases):
    case = next(c for c in ref_cases if c["name"] == "quirk_cycles_forever")
    rows, c = case_inputs(case)
    assert oracle.solve(rows, c, max_pivots=2000).status == oracle.CAP
    o = D.solve(rows, c, max_pivots=2000)
    assert (o.status, o.npiv) == (oracle.NOCONV, 0)


def test_phase1_1000_ends_optimal():
    rows, c = W.phase1_lp(1000, 1000, 0)
    o = D.solve(rows, c, max_pivots=20000)
    assert o.status == oracle.OPTIMAL


def test_a_feasible_row_stays_feasible():
    for seed in range(3):
        for n, m in ((15, 25), (30, 20), (60, 40)):
            rows, c = W.phase1_lp(n, m, seed)
            o = D.solve(rows, c, max_pivots=2000, snapshots=True)
            b = o.snaps[:, : n * (m + 1)].reshape(-1, n, m + 1)[:, :, m]
            assert not ((b[:-1] >= 0) & (b[1:] < 0)).any(), (n, m, seed)
            assert o.status != oracle.CAP


# --------------------------------------------------------------------------- CPU: the C ABI without a device
@pytest.fixture(scope="module")
def native():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native


def test_abi_version_and_rule_constant(native):
    """A new value of the existing rule argument: callers of version 8 are unaffected, so it stays 8."""
    L = native.load()
    text = open(native.os.path.join(native.os.path.dirname(native.HERE), "include", "spx_b200.h")).read()
    assert L.spx_version() == 8 == native.ABI_VERSION
    assert int(HEADER_RULE.search(text).group(1)) == 4 == native.RULE_DANTZIG_BLAND == native.RULES[RULE]
    assert native.RULES["bland"] == 0 == native.RULE_REFERENCE


def test_single_lp_and_sharded_entries_refuse_the_rule(native):
    import ctypes
    L, f, r = native.load(), FAKE, native.RULE_DANTZIG_BLAND
    words = ("SPX_RULE_DANTZIG_BLAND", "spx_solve_batched")
    _refused(L, L.spx_pick(f, f, 4, 2, 16, r, 0, f, f, None), "spx_pick", *words)
    _refused(L, L.spx_solve(f, f, f, f, 4, 2, 16, r, f, f, f, f, None, 1, 0, 0, None, 0, None, None, None),
             "spx_solve", *words)
    wb = L.spx_fused_workspace_bytes(4, 2)
    _refused(L, L.spx_fused_pass(f, f, f, f, 4, 2, 16, r, 1, 0, f, f, wb, f, f, None, None), "spx_fused_pass", *words)
    _refused(L, L.spx_shard_candidate(f, f, 4, 2, 16, 0, r, 1, f, f, None), "spx_shard_candidate", *words)
    _refused(L, L.spx_shard_select(f, 1, f, 4, r, 1, f, f, None, 0, None), "spx_shard_select", *words)
    _refused(L, L.spx_ahead_candidate(f, f, 2 * f, 4, 2, 16, 0, r, f, f, f, None), "spx_ahead_candidate", *words)
    h = ctypes.c_void_p()
    boxes = (ctypes.c_void_p * 1)(f)
    _refused(L, L.spx_shard_open(ctypes.byref(h), 0, 1, 4, 2, 16, 0, r, f, f, f, f, f, f, f, f, None, f, boxes),
             "spx_shard_open", *words)
    _refused(L, L.spx_fshard_open(ctypes.byref(h), 0, 1, 4, 2, 16, 0, r, f, f, f, f, f, f, 1 << 30, f, f, None,
                                  boxes), "spx_fshard_open", *words)
    # 3 stays unknown to the batched entries, and so does 5
    for bad in (3, 5):
        _refused(L, L.spx_solve_batched(f, 1, 4, 2, bad, 8, f, None, f, f, None, None, None, None, None),
                 f"unknown rule {bad}")


def test_simplex_method_refuses_the_rule():
    from simplex_method_solver_b200.simplex import SimplexMethod
    with pytest.raises(ValueError, match="batched.*labels"):
        SimplexMethod(W.CFG1_ROWS, W.CFG1_C, rule=RULE)


# --------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def spx():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("GPU tests need a CUDA device")
    from simplex_method_solver_b200 import _native, batched

    class NS:
        pass
    ns = NS()
    ns.N, ns.L, ns.batched = _native, _native.lib(), batched
    return ns


def check_lp(res, k, T, n, m, cap, what, snaps=False, o=None):
    """LP k of a BatchResult against dantzig_bland_oracle.c: status, npiv, trace, table, labels, x, obj (and
    snapshots)"""
    o = o or D.solve_flat(T, n, m, cap, snapshots=snaps)
    assert (int(res.status[k]), int(res.npiv[k])) == (o.status, o.npiv), (what, n, m, k)
    assert res.trace[k, : o.npiv].tolist() == o.trace.tolist(), (what, n, m, k)
    assert same(res.tables[k], o.table), (what, n, m, k)
    assert res.rowlab[k].tolist() == o.rowlab.tolist() and res.collab[k].tolist() == o.collab.tolist(), (what, k)
    assert same(res.x[k], o.x) and same(res.obj[k], o.obj2), (what, n, m, k)
    if snaps:
        assert same(res.snaps[k, : o.npiv + 1], o.snaps), (what, n, m, k)
    return o


def check_certificates(spx, res, n, m, what):
    """the solver's stop row is the Farkas row of every SPX_INCORRECT LP; a finite SPX_NOCONV LP has a ray"""
    cert = spx.batched.certificate(res)
    for k in range(res.status.shape[0]):
        T = res.tables[k]
        if int(res.status[k]) == oracle.INCORRECT:
            b = T[m: n * (m + 1): m + 1]
            assert int(cert.farkas_row[k]) == int(np.flatnonzero(b < 0)[0]), (what, k)
        elif int(res.status[k]) == oracle.NOCONV and np.isfinite(T).all():
            assert cert.unbounded[k], (what, k)


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,cap,engine", UNIFORM, ids=[f"{n}x{m}" for n, m, _, _ in UNIFORM])
def test_uniform_every_engine(spx, n, m, cap, engine):
    lo = {"auto": 0, "cluster": spx.L.spx_cluster_size(n, m), "global": spx.L.spx_global_min_cluster_size(n, m)}[engine]
    runs = [(engine, 0)] if engine == "auto" else [(engine, S) for S in SIZES if S >= lo]
    flats = uniform_batch(n, m, 8 if n * m < 100_000 else 4, 17 * n + m)
    snaps = n * m <= 2000
    want = [D.solve_flat(flats[k], n, m, cap, snapshots=snaps) for k in range(flats.shape[0])]
    assert any(o.status == oracle.OPTIMAL for o in want)
    for engine, S in runs:
        with cluster_size(spx.L, S):
            res = spx.batched.solve_batched(flats, n, m, max_pivots=cap, rule=RULE, engine=engine, snapshots=snaps)
        for k in range(flats.shape[0]):
            check_lp(res, k, flats[k], n, m, cap, (engine, S), snaps, want[k])
        check_certificates(spx, res, n, m, (engine, S))


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", sorted(nm for nm, (kind, _) in EDGES.items() if kind is not None))
def test_capacity_edges(spx, n, m):
    kind = EDGES[(n, m)][0]
    flats = np.stack(edge_batch(n, m))
    cap = _cap(n, m)
    for engine, S in engine_runs(spx.L, n, m, kind):
        with cluster_size(spx.L, S):
            res = spx.batched.solve_batched(flats, n, m, max_pivots=cap, rule=RULE, engine=engine)
        for k in range(flats.shape[0]):
            check_lp(res, k, flats[k], n, m, cap, (engine, S))


def ragged_mix():
    lps = W.scaled_lps(40, 2) + W.mixed_lps(16, 3)
    lps += [W.phase1_lp(600, 800, 5), W.phase1_lp(300, 300, 0), W.dense_lp(64, 12000, 6),
            scaled(*W.dense_lp(2000, 300, 7), 7)]
    return lps


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["auto", "auto_global"])
def test_ragged_equals_each_lp_alone(spx, engine):
    from simplex_method_solver_b200.batched import kernel_for
    code = spx.batched.ENGINE_CODES[engine]
    lps = [lp for lp in ragged_mix() if spx.L.spx_batched_route(lp[0].shape[0], lp[1].shape[0], code) >= 0]
    caps = [3000 if lp[0].size > 300_000 else 20000 for lp in lps]
    res = spx.batched.solve_ragged(lps, max_pivots=caps, rule=RULE, engine=engine)
    kinds = set()
    for k, (rows, c) in enumerate(lps):
        n, m = rows.shape[0], c.shape[0]
        T = flat_of(rows, c)
        alone = spx.batched.solve_batched(T[None], n, m, max_pivots=caps[k], rule=RULE, engine=engine)
        one = res.lp(k)
        for a in ("status", "npiv", "x", "obj", "tables", "rowlab", "collab"):
            assert same(getattr(one, a), getattr(alone, a)) if getattr(one, a).dtype.kind == "f" else \
                np.array_equal(getattr(one, a), getattr(alone, a)), (engine, k, a)
        check_lp(one, 0, T, n, m, caps[k], ("ragged", engine))
        kinds.add(kernel_for(n, m, engine))
    assert kinds >= {"smem", "cluster"} and (engine == "auto" or "global" in kinds)


def _resume_oracle(table, n, m, rowlab, collab, db, dc, fn, cap):
    import warm_oracle as WO
    T = WO.change(table, n, m, rowlab, collab, db, dc)
    return D.solve_flat(T, n, m, cap, rowlab=rowlab, collab=collab, function=fn)


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,engine", [(11, 7, "auto"), (40, 60, "auto"), (100, 160, "cluster"),
                                        (600, 800, "global")])
def test_capped_and_resumed_and_resolve(spx, n, m, engine):
    B = spx.batched
    flats = uniform_batch(n, m, 4, 5 * n + m)
    cap = 4000
    # capped at K and resumed for K equals capped at 2K (the rule reads only the table and the labels)
    K = 6
    capped = B.solve_batched(flats, n, m, max_pivots=K, rule=RULE, engine=engine)
    cont = B.resolve(capped, flats, max_pivots=K, rule=RULE, engine=engine)
    twice = B.solve_batched(flats, n, m, max_pivots=2 * K, rule=RULE, engine=engine)
    for k in range(4):
        assert int(cont.status[k]) == int(twice.status[k]), k
        assert int(capped.npiv[k]) + int(cont.npiv[k]) == int(twice.npiv[k]), k
        assert same(cont.tables[k], twice.tables[k]) and same(cont.x[k], twice.x[k]), k
        assert np.array_equal(cont.rowlab[k], twice.rowlab[k]) and np.array_equal(cont.collab[k], twice.collab[k])
        o = D.solve_flat(capped.tables[k], n, m, K, rowlab=capped.rowlab[k], collab=capped.collab[k],
                         function=flats[k, n * (m + 1):])
        check_lp(cont, k, None, n, m, K, ("resume", engine), o=o)
    first = B.solve_batched(flats, n, m, max_pivots=cap, rule=RULE, engine=engine)
    rng = np.random.default_rng(n)
    rhs = flats[:, : n * (m + 1)].reshape(4, n, m + 1)[:, :, m] * rng.uniform(0.9, 1.1, (4, n))
    cost = flats[:, n * (m + 1):] * rng.uniform(0.9, 1.1, (4, m))
    old_b = flats[:, : n * (m + 1)].reshape(4, n, m + 1)[:, :, m]
    for new_rhs, new_cost in ((rhs, None), (None, cost)):
        res = B.resolve(first, flats, rhs=new_rhs, cost=new_cost, max_pivots=cap, rule=RULE, engine=engine)
        for k in range(4):
            db = None if new_rhs is None else new_rhs[k] - old_b[k]
            dc = None if new_cost is None else new_cost[k] - flats[k, n * (m + 1):]
            fn = flats[k, n * (m + 1):] if new_cost is None else new_cost[k]
            o = _resume_oracle(first.tables[k], n, m, first.rowlab[k], first.collab[k], db, dc, fn, cap)
            check_lp(res, k, None, n, m, cap, ("resolve", engine), o=o)


@pytest.mark.gpu
def test_non_finite_every_engine(spx):
    """The adversarial LPs (NaN, +-Inf, -0.0, subnormals, huge pivots, overflow) through K4, K7 and K8 at every
    cluster size, uniform and ragged, and tables with NaN / +-Inf in the f row."""
    B = spx.batched
    every = []
    for n, m in SPECIAL_SHAPES:
        lps = special_lps(n, m)
        flats = np.stack([flat_of(rows, c) for _, _, rows, c, _ in lps])
        every += [(n, m, flat_of(rows, c)) for _, _, rows, c, _ in lps]
        want = [D.solve_flat(T, n, m, SPECIAL_CAP) for T in flats]
        for engine, S in SPECIAL_RUNS:
            with cluster_size(spx.L, S):
                res = B.solve_batched(flats, n, m, max_pivots=SPECIAL_CAP, rule=RULE, engine=engine)
            for k in range(flats.shape[0]):
                check_lp(res, k, None, n, m, SPECIAL_CAP, (engine, S), o=want[k])
            check_certificates(spx, res, n, m, (engine, S))
    for _, n, m, T in nonfinite_tables()[-6:]:
        every.append((n, m, T))
        for engine in ("auto", "cluster", "global"):
            res = B.solve_batched(T[None], n, m, max_pivots=40, rule=RULE, engine=engine)
            check_lp(res, 0, T, n, m, 40, ("f row", engine))
    lps = [(T[: n * (m + 1)].reshape(n, m + 1), T[n * (m + 1):]) for n, m, T in every]
    for engine, S in [("auto_global", 0)] + SPECIAL_RUNS:
        with cluster_size(spx.L, S):
            res = B.solve_ragged(lps, max_pivots=SPECIAL_CAP, rule=RULE, engine=engine)
        for k, (n, m, T) in enumerate(every):
            check_lp(res.lp(k), 0, T, n, m, SPECIAL_CAP, ("ragged", engine, S))


@pytest.mark.gpu
def test_golden_cases_on_k4_and_their_certificates(spx, ref_cases):
    """Every golden case on K4 (warp or CTA mode by its shape) equals the statement; the LPs it stops on carry the
    certificates of their status."""
    groups = {}
    for case in ref_cases:
        rows, c = case_inputs(case)
        rows = np.asarray(rows, dtype=np.float64)
        groups.setdefault((rows.shape[0], c.shape[0]), []).append(flat_of(rows, c))
    for (n, m), flats in groups.items():
        if not spx.L.spx_batched_route(n, m, spx.batched.ENGINE_CODES["auto"]) >= 0:
            continue
        flats = np.stack(flats)
        res = spx.batched.solve_batched(flats, n, m, max_pivots=300, rule=RULE)
        for k in range(flats.shape[0]):
            check_lp(res, k, flats[k], n, m, 300, ("golden", n, m))
        check_certificates(spx, res, n, m, ("golden", n, m))


@pytest.mark.gpu
def test_phase1_1000_on_k8_all_optimal(spx):
    flats = np.stack([flat_of(*W.phase1_lp(1000, 1000, s)) for s in range(8)])
    res = spx.batched.solve_batched(flats, 1000, 1000, max_pivots=20000, rule=RULE, engine="global")
    assert (res.status == oracle.OPTIMAL).all(), res.status
    for k in (0, 5):
        check_lp(res, k, flats[k], 1000, 1000, 20000, "phase1 1000")
