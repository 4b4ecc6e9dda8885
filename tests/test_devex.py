"""The devex entering rule (SPX_RULE_DEVEX): its statements and the batched engines that run it.

CPU part: an independent pure-Python statement (devex_model.py) equals the sequential C statement (devex_oracle.c)
bit for bit on the golden cases, seeded dense, phase-1 and scaled families, Klee-Minty and non-finite tables; with
unit weights devex enters where Dantzig does; Klee-Minty n = 10 ends in at most 100 pivots; the C ABI refuses devex
outside the batched entries and without d_x before touching a device.
GPU part: K4 (warp and CTA mode), K7 at every cluster size and K8 at every S under devex, uniform and ragged, at the
capacity edges and on non-finite inputs, resumes and re-solves, bit for bit against devex_oracle.c.
"""
import ctypes
import re

import numpy as np
import pytest

import devex_model as M
import devex_oracle as D
import oracle
from simplex_method_solver_b200 import workloads as W
from test_capacity_edges import (EDGES, SIZES, SPECIAL_CAP, SPECIAL_RUNS, SPECIAL_SHAPES, _cap, edge_batch,
                                 engine_runs, same, special_lps)
from test_cluster_batched import cluster_size
from util import case_inputs, flat_of

HEADER_RULE = re.compile(r"#define SPX_RULE_DEVEX\s+(\d+)")


def scaled(rows, c, seed):
    """rows, c with the units of every x_j changed (column j and c_j times 10^U(-2, 2)), as workloads.scaled_lps"""
    s = 10.0 ** np.random.default_rng(seed + 7).uniform(-2.0, 2.0, c.shape[0])
    rows = np.array(rows, dtype=np.float64)
    rows[:, : c.shape[0]] *= s
    return rows, c * s


def families():
    """(name, rows, c) of the seeded CPU families"""
    out = []
    for seed in range(3):
        for n, m in ((6, 4), (15, 25), (30, 20)):
            for fam in (W.dense_lp, W.phase1_lp):
                rows, c = fam(n, m, seed)
                out.append((f"{fam.__name__}({n},{m},{seed})", rows, c))
                out.append((f"scaled {fam.__name__}({n},{m},{seed})", *scaled(rows, c, seed)))
    out.append(("KM(10)", *W.klee_minty(10)))
    return out


def nonfinite_tables():
    """(name, n, m, flat) of tables with NaN / +-Inf in the f row and in the body"""
    out = [(f"{kind}@{r0}", n, m, flat_of(rows, c)) for n, m in SPECIAL_SHAPES[:2] for kind, r0, rows, c, _ in
           special_lps(n, m)]
    rng = np.random.default_rng(11)
    for q, vals in enumerate(([np.nan], [np.inf], [-np.inf], [np.nan, -np.inf], [-np.inf, -np.inf], [-1e200, -1e-200])):
        rows, c = W.dense_lp(12, 9, 100 + q)
        c[rng.choice(9, len(vals), replace=False)] = vals
        rows[rng.integers(0, 12), rng.integers(0, 9)] = vals[0]
        out.append((f"f{vals}", 12, 9, flat_of(rows, c)))
    return out


def model_equals_oracle(T, n, m, cap, what):
    o = D.solve_flat(T, n, m, cap)
    st, trace, table, rl, cl = M.solve(T, n, m, cap)
    assert (st, len(trace)) == (o.status, o.npiv), what
    assert [tuple(t) for t in o.trace.tolist()] == trace, what
    assert same(np.asarray(table), o.table), what
    assert rl == o.rowlab.tolist() and cl == o.collab.tolist(), what
    return o


# --------------------------------------------------------------------------- CPU: the rule
def test_model_equals_oracle_on_the_golden_cases(ref_cases):
    assert len(ref_cases) == 381
    for case in ref_cases:
        rows, c = case_inputs(case)
        rows = np.asarray(rows, dtype=np.float64)
        model_equals_oracle(flat_of(rows, c), rows.shape[0], rows.shape[1] - 1, 300, case.get("name", case))


def test_model_equals_oracle_on_seeded_and_scaled_families():
    ends = set()
    for name, rows, c in families():
        o = model_equals_oracle(flat_of(rows, c), rows.shape[0], rows.shape[1] - 1, 2000, name)
        ends.add(o.status)
    assert oracle.OPTIMAL in ends


def test_model_equals_oracle_on_non_finite_tables():
    for name, n, m, T in nonfinite_tables():
        model_equals_oracle(T, n, m, 40, name)


def test_unit_weights_enter_where_dantzig_does(ref_cases):
    """With w = 1 the score is f_j^2: on every phase-2 table the reference visits, devex and Dantzig agree."""
    seen = 0
    for case in ref_cases:
        rows, c = case_inputs(case)
        rows = np.asarray(rows, dtype=np.float64)
        n, m = rows.shape[0], rows.shape[1] - 1
        snaps = oracle.solve(rows, c, max_pivots=200, snapshots=True).snaps
        for T in snaps:
            if (T[m: n * (m + 1): m + 1] < 0).any():
                continue
            assert D.pick(T, n, m, np.ones(m)) == oracle.pick(T, n, m, rule="dantzig")
            seen += 1
    assert seen > 381


def test_klee_minty_10_in_at_most_100_pivots():
    rows, c = W.klee_minty(10)
    o = D.solve(rows, c)
    assert o.status == oracle.OPTIMAL and o.npiv <= 100
    assert oracle.solve(rows, c, rule="dantzig").npiv == 1023


def test_scaled_lps_change_units_only():
    base, sc = W.mixed_lps(6, 3), W.scaled_lps(6, 3)
    for (r0, c0), (r1, c1) in zip(base, sc):
        m = c0.shape[0]
        s = c1 / c0
        assert np.all((s >= 0.01) & (s <= 100.0))
        assert np.array_equal(r1[:, m], r0[:, m]) and np.allclose(r1[:, :m], r0[:, :m] * s)


# --------------------------------------------------------------------------- CPU: the C ABI without a device
@pytest.fixture(scope="module")
def native():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native


FAKE = 1 << 20     # a 128-byte aligned address no call below dereferences


def _refused(L, rc, *words):
    msg = L.spx_last_error().decode()
    assert rc == -2, msg
    for w in words:
        assert w in msg, msg


def test_abi_version_and_rule_constant(native):
    """Devex is a new value of the existing rule argument: callers of version 8 are unaffected, so it stays 8."""
    L = native.load()
    text = open(native.os.path.join(native.os.path.dirname(native.HERE), "include", "spx_b200.h")).read()
    assert L.spx_version() == 8 == native.ABI_VERSION
    assert int(HEADER_RULE.search(text).group(1)) == 2 == native.RULE_DEVEX == native.RULES["devex"]


def test_single_lp_and_sharded_entries_refuse_devex(native):
    L, f = native.load(), FAKE
    _refused(L, L.spx_pick(f, f, 4, 2, 16, 2, 0, f, f, None), "spx_pick", "spx_solve_batched")
    _refused(L, L.spx_solve(f, f, f, f, 4, 2, 16, 2, f, f, f, f, None, 1, 0, 0, None, 0, None, None, None),
             "spx_solve", "batched")
    wb = L.spx_fused_workspace_bytes(4, 2)
    _refused(L, L.spx_fused_pass(f, f, f, f, 4, 2, 16, 2, 1, 0, f, f, wb, f, f, None, None), "spx_fused_pass",
             "batched")
    _refused(L, L.spx_shard_candidate(f, f, 4, 2, 16, 0, 2, 1, f, f, None), "spx_shard_candidate", "batched")
    _refused(L, L.spx_shard_select(f, 1, f, 4, 2, 1, f, f, None, 0, None), "spx_shard_select", "batched")
    _refused(L, L.spx_ahead_candidate(f, f, 2 * f, 4, 2, 16, 0, 2, f, f, f, None), "spx_ahead_candidate", "batched")
    h = ctypes.c_void_p()
    boxes = (ctypes.c_void_p * 1)(f)
    _refused(L, L.spx_shard_open(ctypes.byref(h), 0, 1, 4, 2, 16, 0, 2, f, f, f, f, f, f, f, f, None, f, boxes),
             "spx_shard_open", "batched")
    _refused(L, L.spx_fshard_open(ctypes.byref(h), 0, 1, 4, 2, 16, 0, 2, f, f, f, f, f, f, 1 << 30, f, f, None,
                                  boxes), "spx_fshard_open", "batched")


def test_batched_entries_refuse_devex_without_x(native):
    L, f = native.load(), FAKE
    for entry in ("spx_solve_batched", "spx_solve_batched_cluster", "spx_solve_batched_global"):
        _refused(L, getattr(L, entry)(f, 1, 4, 2, 2, 8, None, None, f, f, None, None, None, None, None), entry, "d_x")
    _refused(L, L.spx_warm_solve_batched(native.ENGINE_AUTO, f, 1, 4, 2, 2, 8, None, None, None, f, f, f, f, None,
                                         None, None), "spx_warm_solve_batched", "d_x")
    from simplex_method_solver_b200.batched import ragged_plan
    plan = ragged_plan([(4, 2), (30, 30)], 8).plan
    _refused(L, L.spx_solve_batched_ragged(f, plan.ctypes.data, f, 2, None, None, f, f, None, None, None, None, None),
             "spx_solve_batched_ragged", "d_x")
    _refused(L, L.spx_warm_solve_ragged(f, plan.ctypes.data, f, 2, None, None, None, f, f, f, f, None, None, None),
             "spx_warm_solve_ragged", "d_x")
    _refused(L, L.spx_solve_batched(f, 1, 4, 2, 3, 8, f, None, f, f, None, None, None, None, None), "unknown rule 3")


def test_simplex_method_refuses_devex():
    from simplex_method_solver_b200.simplex import SimplexMethod
    with pytest.raises(ValueError, match="batched"):
        SimplexMethod(W.CFG1_ROWS, W.CFG1_C, rule="devex")


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
    """LP k of a BatchResult against devex_oracle.c: status, npiv, trace, table, labels, x, obj (and snapshots)"""
    o = o or D.solve_flat(T, n, m, cap, snapshots=snaps)
    assert (int(res.status[k]), int(res.npiv[k])) == (o.status, o.npiv), (what, n, m, k)
    assert res.trace[k, : o.npiv].tolist() == o.trace.tolist(), (what, n, m, k)
    assert same(res.tables[k], o.table), (what, n, m, k)
    assert res.rowlab[k].tolist() == o.rowlab.tolist() and res.collab[k].tolist() == o.collab.tolist(), (what, k)
    assert same(res.x[k], o.x) and same(res.obj[k], o.obj2), (what, n, m, k)
    if snaps:
        assert same(res.snaps[k, : o.npiv + 1], o.snaps), (what, n, m, k)
    return o


def uniform_batch(n, m, B, seed):
    """golden-like dense and phase-1 LPs, plain and scaled"""
    out = []
    for q in range(B):
        rows, c = (W.dense_lp if q % 2 else W.phase1_lp)(n, m, seed + q)
        out.append(flat_of(*(scaled(rows, c, seed + q) if q % 4 >= 2 else (rows, c))))
    return np.stack(out)


# (n, m, cap, engine): K4 warp mode, K4 CTA mode, K7 at every cluster size that holds the LP, K8 at every S
UNIFORM = [(8, 2, 64, "auto"), (11, 7, 100, "auto"), (20, 20, 400, "auto"), (40, 60, 2000, "auto"),
           (100, 160, 4000, "cluster"), (300, 400, 4000, "cluster"), (600, 800, 4000, "global")]


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,cap,engine", UNIFORM, ids=[f"{n}x{m}" for n, m, _, _ in UNIFORM])
def test_devex_uniform_every_engine(spx, n, m, cap, engine):
    lo = {"auto": 0, "cluster": spx.L.spx_cluster_size(n, m), "global": spx.L.spx_global_min_cluster_size(n, m)}[engine]
    runs = [(engine, 0)] if engine == "auto" else [(engine, S) for S in SIZES if S >= lo]
    flats = uniform_batch(n, m, 8 if n * m < 100_000 else 4, 17 * n + m)
    snaps = n * m <= 2000
    want = [D.solve_flat(flats[k], n, m, cap, snapshots=snaps) for k in range(flats.shape[0])]
    assert any(o.status == oracle.OPTIMAL for o in want)
    for engine, S in runs:
        with cluster_size(spx.L, S):
            res = spx.batched.solve_batched(flats, n, m, max_pivots=cap, rule="devex", engine=engine,
                                            snapshots=snaps)
        for k in range(flats.shape[0]):
            check_lp(res, k, flats[k], n, m, cap, (engine, S), snaps, want[k])


@pytest.mark.gpu
def test_devex_klee_minty_on_k4_cta_mode(spx):
    rows, c = W.klee_minty(15)
    T = flat_of(rows, c)[None]
    res = spx.batched.solve_batched(T, 15, 15, max_pivots=1000, rule="devex")
    o = check_lp(res, 0, T[0], 15, 15, 1000, "KM(15)")
    assert o.status == oracle.OPTIMAL and o.npiv == 143


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", sorted(nm for nm, (kind, _) in EDGES.items() if kind is not None))
def test_devex_capacity_edges(spx, n, m):
    kind = EDGES[(n, m)][0]
    flats = np.stack(edge_batch(n, m))
    cap = _cap(n, m)
    for engine, S in engine_runs(spx.L, n, m, kind):
        with cluster_size(spx.L, S):
            res = spx.batched.solve_batched(flats, n, m, max_pivots=cap, rule="devex", engine=engine)
        for k in range(flats.shape[0]):
            check_lp(res, k, flats[k], n, m, cap, (engine, S))


def ragged_mix():
    lps = W.scaled_lps(48, 2)
    lps += [scaled(*W.phase1_lp(600, 800, 5), 5), W.dense_lp(64, 12000, 6), scaled(*W.dense_lp(2000, 300, 7), 7)]
    return lps


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["auto", "auto_global"])
def test_devex_ragged_equals_each_lp_alone(spx, engine):
    from simplex_method_solver_b200.batched import kernel_for
    code = spx.batched.ENGINE_CODES[engine]
    lps = [lp for lp in ragged_mix() if spx.L.spx_batched_route(lp[0].shape[0], lp[1].shape[0], code) >= 0]
    caps = [3000 if lp[0].size > 300_000 else 20000 for lp in lps]
    res = spx.batched.solve_ragged(lps, max_pivots=caps, rule="devex", engine=engine)
    kinds = set()
    for k, (rows, c) in enumerate(lps):
        n, m = rows.shape[0], c.shape[0]
        T = flat_of(rows, c)
        alone = spx.batched.solve_batched(T[None], n, m, max_pivots=caps[k], rule="devex", engine=engine)
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
def test_devex_resolve_uniform(spx, n, m, engine):
    B = spx.batched
    flats = uniform_batch(n, m, 4, 5 * n + m)
    cap = 4000
    first = B.solve_batched(flats, n, m, max_pivots=cap, rule="devex", engine=engine)
    rng = np.random.default_rng(n)
    rhs = flats[:, : n * (m + 1)].reshape(4, n, m + 1)[:, :, m] * rng.uniform(0.9, 1.1, (4, n))
    cost = flats[:, n * (m + 1):] * rng.uniform(0.9, 1.1, (4, m))
    res = B.resolve(first, flats, rhs=rhs, cost=cost, max_pivots=cap, rule="devex", engine=engine)
    old_b = flats[:, : n * (m + 1)].reshape(4, n, m + 1)[:, :, m]
    for k in range(4):
        o = _resume_oracle(first.tables[k], n, m, first.rowlab[k], first.collab[k], rhs[k] - old_b[k],
                           cost[k] - flats[k, n * (m + 1):], cost[k], cap)
        check_lp(res, k, None, n, m, cap, ("resolve", engine), o=o)
    # a capped solve resumed: the oracle's devex solve from the capped table with unit weights
    capped = B.solve_batched(flats, n, m, max_pivots=3, rule="devex", engine=engine)
    cont = B.resolve(capped, flats, max_pivots=cap, rule="devex", engine=engine)
    for k in range(4):
        o = D.solve_flat(capped.tables[k], n, m, cap, rowlab=capped.rowlab[k], collab=capped.collab[k],
                         function=flats[k, n * (m + 1):])
        check_lp(cont, k, None, n, m, cap, ("resume", engine), o=o)


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["auto", "auto_global"])
def test_devex_resolve_ragged(spx, engine):
    B = spx.batched
    lps = W.scaled_lps(24, 4)
    if engine == "auto_global":
        lps.append(W.phase1_lp(600, 800, 9))
    cap = 20000
    first = B.solve_ragged(lps, max_pivots=cap, rule="devex", engine=engine)
    rng = np.random.default_rng(3)
    rhs = [rows[:, -1] * rng.uniform(0.9, 1.1, rows.shape[0]) for rows, _ in lps]
    cost = [c * rng.uniform(0.9, 1.1, c.shape[0]) for _, c in lps]
    res = B.resolve(first, lps, rhs=rhs, cost=cost, max_pivots=cap, rule="devex", engine=engine)
    for k, (rows, c) in enumerate(lps):
        n, m = rows.shape[0], c.shape[0]
        f0 = first.lp(k)
        o = _resume_oracle(f0.tables[0], n, m, f0.rowlab[0], f0.collab[0], rhs[k] - rows[:, m], cost[k] - c,
                           cost[k], cap)
        check_lp(res.lp(k), 0, None, n, m, cap, ("ragged resolve", engine), o=o)


@pytest.mark.gpu
def test_devex_non_finite_every_engine(spx):
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
                res = B.solve_batched(flats, n, m, max_pivots=SPECIAL_CAP, rule="devex", engine=engine)
            for k in range(flats.shape[0]):
                check_lp(res, k, None, n, m, SPECIAL_CAP, (engine, S), o=want[k])
    for _, n, m, T in nonfinite_tables()[-6:]:
        every.append((n, m, T))
        for engine in ("auto", "cluster", "global"):
            res = B.solve_batched(T[None], n, m, max_pivots=40, rule="devex", engine=engine)
            check_lp(res, 0, T, n, m, 40, ("f row", engine))
    lps = [(T[: n * (m + 1)].reshape(n, m + 1), T[n * (m + 1):]) for n, m, T in every]
    for engine, S in [("auto_global", 0)] + SPECIAL_RUNS:
        with cluster_size(spx.L, S):
            res = B.solve_ragged(lps, max_pivots=SPECIAL_CAP, rule="devex", engine=engine)
        for k, (n, m, T) in enumerate(every):
            check_lp(res.lp(k), 0, T, n, m, SPECIAL_CAP, ("ragged", engine, S))
