"""Ragged batches with K8: engine="global" (every LP on K8) and engine="auto_global" (K4, else K7, else K8) in
spx_ragged_plan / spx_solve_batched_ragged / batched.solve_ragged, and SimplexMethod(engine="global").

CPU part: plan routing and order over every class, the auto_global plan against the auto plan, the 12-launch bound,
forced cluster sizes (no device), validation and error texts, kernel_for's edges, the sharded pass-through, the
SimplexMethod engine check.
GPU part: both golden sets in one call at every forced S; a mixed K4/K7/K8 batch against the oracle and against
per-LP solve_batched; a band above 2^24 cells; snapshots; launch counts; batch order and mates; reuse and the empty
batch; the default cluster size of a K8 launch; get_solution() on K8.
"""
import numpy as np
import pytest

import oracle
from simplex_method_solver_b200 import workloads as W
from test_cluster_batched import _family, cluster_size
from test_global_batched import expected_min_size
from test_ragged_batched import _check_case, _golden_lps, _plan_raw, random_shapes
from util import END_TO_STATUS, bits, flat_of, label_codes, table_sha

SIZES = (1, 2, 4, 8, 16)
# one K8 shape per S_min: 1 x m with m above K7's 9,499 columns, and 600 x 800 (S_min 1)
K8_BY_SMIN = {1: (600, 800), 2: (64, 12000), 4: (1, 13000), 8: (1, 13800), 16: (1, 14000)}


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native.load()


def cells_of(n, m):
    return n * (m + 1) + m


def expected_class(L, n, m, engine):
    """(kind, planned S) of an LP under `engine`, from the uniform entries' own rules."""
    from simplex_method_solver_b200.batched import kernel_for
    forced = L.spx_get_option(16)
    kind = kernel_for(n, m, engine)
    if kind == "smem":
        return ("warp" if cells_of(n, m) <= 96 else "cta"), 1
    if kind == "cluster":
        return "cluster", (forced or L.spx_cluster_size(n, m))
    return "global", (forced or L.spx_global_min_cluster_size(n, m))


def k8_shapes(rng, B):
    """Shapes above K7's capacity: tall / wide at m <= 2,000 (S_min 1 or 2) and 1..200 x 9,500..14,177."""
    out = []
    for _ in range(B):
        if rng.integers(0, 2):
            out.append((int(rng.integers(529, 4000)), int(rng.integers(600, 2001))))
        else:
            out.append((int(rng.integers(1, 200)), int(rng.integers(9500, 14178))))
    return out


# --------------------------------------------------------------------------- CPU
def test_k8_shapes_have_the_intended_min_size(lib):
    for S, (n, m) in K8_BY_SMIN.items():
        assert lib.spx_cluster_size(n, m) == 0 and lib.spx_global_min_cluster_size(n, m) == S == expected_min_size(n, m)


@pytest.mark.parametrize("engine", ["global", "auto_global"])
def test_plan_routing_order_and_launch_count(lib, engine):
    from simplex_method_solver_b200.batched import kernels_for, ragged_plan
    rng = np.random.default_rng(7)
    shapes = random_shapes(rng, 300) + k8_shapes(rng, 60) + list(K8_BY_SMIN.values())
    shapes += shapes[:5] + shapes[-5:]                     # equal cells: ties by index
    p = ragged_plan(shapes, 10, engine)
    seen, kinds = [], []
    for la in p.launches:
        idx = la["lps"].tolist()
        seen += idx
        kinds.append((la["kind"], la["S"]))
        for k in idx:
            assert expected_class(lib, *shapes[k], engine) == (la["kind"], la["S"]), (k, shapes[k])
        key = [(-cells_of(*shapes[k]), k) for k in idx]
        assert key == sorted(key), "largest first, ties by batch index"
    assert sorted(seen) == list(range(len(shapes)))
    classes = {expected_class(lib, n, m, engine) for n, m in shapes}
    assert len(p.launches) == len(classes) and set(kinds) == classes
    rank = {"warp": 0, "cta": 1, "cluster": 2, "global": 3}
    assert kinds == sorted(kinds, key=lambda c: (rank[c[0]], c[1])), "warp, CTA, K7 by S, K8 by S_min"
    if engine == "global":
        assert {c[0] for c in kinds} == {"global"} and {c[1] for c in kinds} == set(SIZES)
    else:
        assert {c[0] for c in kinds} == {"warp", "cta", "cluster", "global"}
    assert kernels_for(shapes, engine) == [{"warp": "smem", "cta": "smem"}.get(c[0], c[0])
                                           for c in (expected_class(lib, n, m, engine) for n, m in shapes)]


def test_auto_global_plan_equals_auto_plan_where_auto_accepts(lib):
    from simplex_method_solver_b200.batched import ragged_plan
    rng = np.random.default_rng(8)
    for B in (1, 5, 200):
        shapes = random_shapes(rng, B)
        caps = rng.integers(0, 500, B)
        a, g = ragged_plan(shapes, caps, "auto"), ragged_plan(shapes, caps, "auto_global")
        assert a.lps.tobytes() == g.lps.tobytes() and a.totals.tolist() == g.totals.tolist()
        assert len(a.launches) == len(g.launches)
        for la, lg in zip(a.launches, g.launches):
            assert {k: v for k, v in la.items() if k != "lps"} == {k: v for k, v in lg.items() if k != "lps"}
            assert la["lps"].tolist() == lg["lps"].tolist()


def test_twelve_launches(lib):
    from simplex_method_solver_b200.batched import ragged_plan
    k7 = [(100, 100), (128, 256), (256, 300), (256, 512), (400, 800)]          # S = 1, 2, 4, 8, 16
    shapes = [(8, 2), (20, 20)] + k7 + [K8_BY_SMIN[S] for S in SIZES]
    p = ragged_plan(shapes, 5, "auto_global")
    assert len(p.launches) == 12
    assert [(la["kind"], la["S"]) for la in p.launches] == (
        [("warp", 1), ("cta", 1)] + [("cluster", S) for S in SIZES] + [("global", S) for S in SIZES])
    assert [la["lps"].tolist() for la in p.launches] == [[k] for k in range(12)]
    for k, la in enumerate(p.launches[7:]):
        n, m = shapes[7 + k]
        R, Q = -(-n // la["S"]), -(-m // la["S"])
        assert la["smem"] == 8 * (2 * m + 1 + R) + 4 * (R + Q) and la["threads"] == 512


def test_forced_cluster_size_needs_no_device(lib):
    from simplex_method_solver_b200.batched import ragged_plan
    k8 = [(600, 800), (2000, 300), (1000, 1000), (64, 12000), (1, 13000), (1, 13800), (1, 14000)]
    for S in SIZES:
        with cluster_size(lib, S):
            fits = [(n, m) for n, m in k8 if lib.spx_global_min_cluster_size(n, m) <= S]
            for engine in ("global", "auto_global"):
                shapes = [(8, 2), (30, 30)] + fits
                p = ragged_plan(shapes, 10, engine)
                got = [(la["kind"], la["S"]) for la in p.launches]
                k8_launches = [g for g in got if g[0] == "global"]
                assert k8_launches == [("global", S)], (S, engine, got)
                rc, err, plan = _plan_raw(lib, [(n, m, 10) for n, m in shapes], engine={"global": 4, "auto_global": 5}[engine])
                assert rc == 0
                for q, (kind, s) in enumerate(got):
                    assert lib.spx_ragged_cluster_size(plan.ctypes.data, q) == s
            bad = next(((n, m) for n, m in k8 if lib.spx_global_min_cluster_size(n, m) > S), None)
            if bad is not None:
                rc, err, _ = _plan_raw(lib, [(8, 2, 5), (600, 800, 5), (bad[0], bad[1], 5)], engine=5)
                assert rc < 0, S
                assert (f"LP 2: a {bad[0]} x {bad[1]} LP does not fit a cluster of SPX_OPT_CLUSTER_SIZE = {S} CTAs"
                        .encode() in err), err


def test_cluster_size_query_without_a_device_for_planned_sizes(lib):
    rc, _, plan = _plan_raw(lib, [(8, 2, 5), (20, 20, 5), (100, 100, 5), (400, 800, 5)])
    assert rc == 0
    assert [lib.spx_ragged_cluster_size(plan.ctypes.data, q) for q in range(4)] == [1, 1, 1, 16]
    assert lib.spx_ragged_cluster_size(plan.ctypes.data, 4) == -1 and b"launch 4" in lib.spx_last_error()
    assert lib.spx_ragged_cluster_size(plan.ctypes.data, -1) == -1
    assert lib.spx_ragged_cluster_size(None, 0) == -1


def test_cluster_size_query_refuses_an_inconsistent_plan_header(lib):
    from simplex_method_solver_b200.batched import _HEADER, _LAUNCH
    rc, _, plan = _plan_raw(lib, [(8, 2, 5), (400, 800, 5)], engine=5)
    assert rc == 0 and lib.spx_ragged_cluster_size(plan.ctypes.data, 0) == 1
    count = _HEADER.fields["launch"][1] + _LAUNCH.fields["count"][1]       # launch[0].count
    plan[count: count + 8].view("<i8")[0] += 1                             # the launches no longer cover B LPs
    assert lib.spx_ragged_cluster_size(plan.ctypes.data, 0) == -1
    assert b"inconsistent plan" in lib.spx_last_error()


def test_plan_validation(lib):
    rc, err, _ = _plan_raw(lib, [(8, 2, 5), (600, 800, 5), (263857, 2000, 5)], engine=5)
    assert rc < 0 and b"LP 2: a 263857 x 2000 LP exceeds the shared memory of one cluster" in err, err
    assert b"230400 bytes" in err
    rc, err, _ = _plan_raw(lib, [(1, 14178, 5)], engine=4)
    assert rc < 0 and b"LP 0: a 1 x 14178 LP exceeds" in err and b"230400 bytes" in err, err
    for engine in (3, 6, -1):
        rc, err, _ = _plan_raw(lib, [(8, 2, 5)], engine=engine)
        assert rc < 0 and b"unknown engine %d" % engine in err, err
    # engine auto keeps its error above K7's capacity
    rc, err, _ = _plan_raw(lib, [(8, 2, 5), (600, 800, 5)], engine=0)
    assert rc < 0 and b"LP 1: a 600 x 800 LP exceeds one cluster" in err, err
    # a plan of an older ABI is refused by the solve entry and by the cluster-size query
    rc, _, plan = _plan_raw(lib, [(8, 2, 5), (600, 800, 5)], engine=5)
    assert rc == 0
    old = plan.copy()
    old[4:8] = np.frombuffer(np.int32(7).tobytes(), np.uint8)
    fake = 4096
    assert lib.spx_solve_batched_ragged(fake, old.ctypes.data, fake, 0, None, None, fake, fake, None, None, None, None,
                                        None) < 0
    assert b"ABI version" in lib.spx_last_error()
    assert lib.spx_ragged_cluster_size(old.ctypes.data, 0) == -1 and b"ABI version" in lib.spx_last_error()
    assert lib.spx_version() == 8


def test_python_routing(lib):
    from simplex_method_solver_b200.batched import ENGINE_CODES, ENGINES, kernel_for, kernels_for, ragged_plan
    assert "auto_global" in ENGINES and ENGINE_CODES["global"] == 4 and ENGINE_CODES["auto_global"] == 5
    edges = {(72, 136): "smem", (1, 5000): "cluster",                      # 10,000 / 10,001 cells
             (528, 800): "cluster", (529, 800): "global", (1, 9499): "cluster", (1, 9500): "global",
             (15866, 2000): "global", (263856, 2000): "global", (1, 14177): "global"}
    assert cells_of(72, 136) == 10000 and cells_of(1, 5000) == 10001
    for (n, m), kind in edges.items():
        assert kernel_for(n, m, "auto_global") == kind, (n, m)
    with pytest.raises(ValueError, match="at most n = 263856 rows"):
        kernel_for(263857, 2000, "auto_global")
    with pytest.raises(ValueError, match="at most 14177 columns"):
        kernel_for(1, 14178, "auto_global")
    with pytest.raises(ValueError, match="at most n = 528 rows"):
        kernel_for(529, 800)                                # "auto" is unchanged
    with pytest.raises(ValueError, match=r"^LP 2: .*at most n = 263856 rows"):
        kernels_for([(8, 2), (600, 800), (263857, 2000)], "auto_global")
    with pytest.raises(ValueError, match="unknown engine"):
        ragged_plan([(8, 2)], 5, "bogus")
    p = ragged_plan([(600, 800), (64, 12000)], 5, "global")
    assert [(la["kind"], la["S"]) for la in p.launches] == [("global", 1), ("global", 2)]


def test_sharded_ragged_passes_the_engine_on():
    from simplex_method_solver_b200.parallel import solve_ragged_sharded
    lps = [W.dense_lp(4, 3, s) for s in range(6)] + [W.dense_lp(600, 800, 0)]
    calls = []

    def stand_in(part, max_pivots, rule, trace, snapshots, device, engine):
        calls.append((len(part), engine))
        return "result"
    for rank in range(2):
        start, count, res = solve_ragged_sharded(lps, max_pivots=7, rank=rank, world=2, solver=stand_in,
                                                 engine="auto_global")
        assert res == "result" and calls[-1] == (count, "auto_global")


def test_simplex_method_accepts_engine_global():
    from simplex_method_solver_b200 import _native as N
    from simplex_method_solver_b200.simplex import SimplexMethod
    rows, c = W.dense_lp(4, 3, 0)
    with pytest.raises(ValueError, match="unknown engine 'bogus'"):
        SimplexMethod(rows, c, engine="bogus")
    try:
        SimplexMethod(rows, c, engine="global")
    except N.NativeUnavailable:
        pass                                               # no device here: the engine check passed first


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
    ns.N, ns.L, ns.batched, ns.torch = _native, _native.lib(), batched, torch
    return ns


@pytest.mark.gpu
@pytest.mark.parametrize("S", SIZES)
def test_golden_sets_in_one_global_call(spx, ref_cases, dantzig_cases, S):
    lps, caps = _golden_lps(ref_cases)
    with cluster_size(spx.L, S):
        db = spx.batched.DeviceRaggedBatch([(r.shape[0], c.shape[0]) for r, c in lps], caps, engine="global")
        assert db.launches == 1 and set(db.kernels) == {"global"} and db.cluster_sizes == [S]
        res = spx.batched.solve_ragged(lps, max_pivots=caps, engine="global")
    for k, case in enumerate(ref_cases):
        _check_case(res.lp(k), case, lps[k][1].shape[0])
    lps, caps = _golden_lps(dantzig_cases)
    with cluster_size(spx.L, S):
        res = spx.batched.solve_ragged(lps, max_pivots=caps, rule="dantzig", engine="global")
    for k, case in enumerate(dantzig_cases):
        one, m = res.lp(k), lps[k][1].shape[0]
        assert int(one.status[0]) == END_TO_STATUS[case["end"]], case["name"]
        assert one.trace[0, : int(one.npiv[0])].tolist() == case["trace"], case["name"]
        assert table_sha(one.tables[0]) == case["final_table_sha256"], case["name"]
        assert one.rowlab[0].tolist() == label_codes(case["row_labels"][:-1], m), case["name"]
        assert one.collab[0].tolist() == label_codes(case["column_labels"][:-1], m), case["name"]


SMALL = [(4, 2), (11, 6), (30, 30), (99, 99), (100, 100), (128, 256), (400, 800)]
LARGE = [(600, 800), (2000, 300), (64, 12000)]
FAMILIES = ("dense", "phase1", "zeros", "incorrect", "noconv")


def _mixed_large(seed):
    """K4 and K7 LPs of every family, then the five families at each K8 shape and a cap hit (cap 1 on a 600 x 800)."""
    lps, caps = [], []
    for q, (n, m) in enumerate(SMALL):
        for f, kind in enumerate(FAMILIES[:3]):
            lps.append(_family(kind, n, m, seed + 10 * q + f))
            caps.append(3000)
    for q, (n, m) in enumerate(LARGE):
        for f, kind in enumerate(FAMILIES):
            lps.append(_family(kind, n, m, seed + 100 + 10 * q + f))
            caps.append(3000)
    lps.append(_family("phase1", 600, 800, seed + 500))
    caps.append(1)
    return lps, caps


def _same(a_res, b_res, what):
    for f, a, b in zip(a_res._fields, a_res, b_res):
        if a is None:
            assert b is None, (what, f)
            continue
        assert a.shape == b.shape and a.dtype == b.dtype, (what, f, a.shape, b.shape)
        assert a.tobytes() == b.tobytes(), (what, f)


@pytest.mark.gpu
def test_auto_global_batch_against_oracle_and_per_lp(spx):
    lps, caps = _mixed_large(1)
    shapes = [(r.shape[0], c.shape[0]) for r, c in lps]
    db = spx.batched.DeviceRaggedBatch(shapes, caps, engine="auto_global")
    assert {k for k in db.kernels} == {"smem", "cluster", "global"}
    assert [la["kind"] for la in db.plan.launches].count("global") == 2          # S_min 1 and 2
    spx.L.spx_launch_count(1)
    res = spx.batched.solve_ragged(lps, max_pivots=caps, engine="auto_global")
    assert spx.L.spx_launch_count(1) == db.launches
    ends = set()
    for k, (rows, c) in enumerate(lps):
        n, m = shapes[k]
        o = oracle.solve_flat(flat_of(rows, c), n, m, max_pivots=caps[k])
        one = res.lp(k)
        ends.add(o.status)
        assert (int(one.status[0]), int(one.npiv[0])) == (o.status, o.npiv), (k, n, m)
        assert one.trace[0, : o.npiv].tolist() == o.trace.tolist(), k
        assert np.array_equal(bits(one.tables[0]), bits(o.table)), k
        assert one.rowlab[0].tolist() == o.rowlab.tolist() and one.collab[0].tolist() == o.collab.tolist(), k
        assert np.array_equal(bits(one.x[0]), bits(o.x)) and bits(one.obj[0]) == bits(o.obj2), k
        alone = spx.batched.solve_batched(flat_of(rows, c)[None, :], n, m, max_pivots=caps[k], engine="auto_global")
        _same(alone, one, k)
    assert {oracle.CAP, oracle.OPTIMAL, oracle.INCORRECT, oracle.NOCONV} <= ends


@pytest.mark.gpu
def test_band_above_2_pow_24_cells_in_a_ragged_batch(spx):
    n, m, cap = 9000, 2000, 30
    assert n * (m + 1) > 1 << 24
    lps = [W.dense_lp(8, 2, 1), W.phase1_lp(n, m, 3), W.dense_lp(600, 800, 2)]
    caps = [20, cap, 25]
    with cluster_size(spx.L, 1):
        res = spx.batched.solve_ragged(lps, max_pivots=caps, engine="auto_global")
    for k, (rows, c) in enumerate(lps):
        o = oracle.solve_flat(flat_of(rows, c), rows.shape[0], c.shape[0], max_pivots=caps[k])
        one = res.lp(k)
        assert (int(one.status[0]), int(one.npiv[0])) == (o.status, o.npiv), k
        assert one.trace[0, : o.npiv].tolist() == o.trace.tolist(), k
        assert np.array_equal(bits(one.tables[0]), bits(o.table)), k
        assert np.array_equal(bits(one.x[0]), bits(o.x)) and one.collab[0].tolist() == o.collab.tolist(), k
    assert int(res.npiv[1]) == cap


@pytest.mark.gpu
def test_snapshots_of_k8_lps(spx):
    lps = [W.phase1_lp(4, 2, 1), W.phase1_lp(100, 100, 2), W.phase1_lp(600, 800, 3), W.phase1_lp(2000, 300, 4),
           W.phase1_lp(30, 30, 5)]
    caps = [6, 12, 8, 0, 20]
    for engine in ("auto_global", "global"):
        res = spx.batched.solve_ragged(lps, max_pivots=caps, snapshots=True, engine=engine)
        for k, (rows, c) in enumerate(lps):
            n, m = rows.shape[0], c.shape[0]
            o = oracle.solve_flat(flat_of(rows, c), n, m, max_pivots=caps[k], snapshots=True)
            one = res.lp(k)
            assert int(one.npiv[0]) == o.npiv and one.snaps.shape == (1, caps[k] + 1, cells_of(n, m))
            assert np.array_equal(bits(one.snaps[0, : o.npiv + 1]), bits(o.snaps)), (engine, k)


@pytest.mark.gpu
def test_independence_from_order_and_mates(spx):
    lps, caps = _mixed_large(2)
    caps = [min(c, 400) for c in caps]
    res = spx.batched.solve_ragged(lps, max_pivots=caps, engine="auto_global")
    perm = np.random.default_rng(3).permutation(len(lps))
    res2 = spx.batched.solve_ragged([lps[q] for q in perm], max_pivots=[caps[q] for q in perm], engine="auto_global")
    for j, q in enumerate(perm):
        _same(res.lp(int(q)), res2.lp(j), (j, q))
    keep = [k for k in range(len(lps)) if k % 3 == 1]                 # other mates, other launch sizes
    res3 = spx.batched.solve_ragged([lps[k] for k in keep], max_pivots=[caps[k] for k in keep], engine="auto_global")
    for j, k in enumerate(keep):
        _same(res.lp(k), res3.lp(j), (j, k))


@pytest.mark.gpu
def test_reuse_empty_and_launch_counts(spx):
    shapes = [(8, 2), (100, 100), (600, 800), (64, 12000)]
    db = spx.batched.DeviceRaggedBatch(shapes, [50, 2000, 300, 300], engine="auto_global")
    assert db.kernels == ["smem", "cluster", "global", "global"] and db.launches == 4
    assert len(db.cluster_sizes) == 4 and db.cluster_sizes[:2] == [1, 1]
    for seed in (1, 2):
        lps = [W.phase1_lp(n, m, seed * 10 + s) for s, (n, m) in enumerate(shapes)]
        db.upload(np.concatenate([flat_of(r, c) for r, c in lps]))
        spx.L.spx_launch_count(1)
        db.run(spx.N.RULE_REFERENCE)
        res = db.result()
        assert spx.L.spx_launch_count(1) == 4
        for k, (rows, c) in enumerate(lps):
            o = oracle.solve_flat(flat_of(rows, c), rows.shape[0], c.shape[0], max_pivots=db.caps[k])
            assert (int(res.status[k]), int(res.npiv[k])) == (o.status, o.npiv), (seed, k)
            assert np.array_equal(bits(res.lp(k).tables[0]), bits(o.table)), (seed, k)
    for engine in ("global", "auto_global"):
        empty = spx.batched.solve_ragged([], max_pivots=10, engine=engine)
        assert empty.status.shape == (0,) and empty.tables.shape == (0,) and empty.shapes.shape == (0, 3)
    with pytest.raises(ValueError, match=r"^LP 1: .*at most 14177 columns"):
        spx.batched.solve_ragged([W.dense_lp(4, 2, 0), W.dense_lp(1, 14178, 0)], engine="auto_global")


@pytest.mark.gpu
def test_default_cluster_size_of_a_single_shape_launch(spx):
    for (n, m), count in (((600, 800), 1), ((600, 800), 64), ((1000, 1000), 32), ((64, 12000), 64),
                          ((2000, 300), 8), ((1000, 2000), 16), ((600, 800), 300)):
        db = spx.batched.DeviceRaggedBatch([(n, m)] * count, 0, engine="global")
        assert db.launches == 1
        assert db.cluster_sizes == [spx.L.spx_global_cluster_size(n, m, count)], (n, m, count)


def _infos(infos):
    from simplex_method_solver_b200.simplex import Error
    return [str(i) if isinstance(i, Error) else (i.row, i.column, i.table, i.i, i.j, i.x1, i.x2, i.optimum)
            for i in infos]


@pytest.mark.gpu
def test_get_solution_on_k8(spx):
    from simplex_method_solver_b200.simplex import SimplexMethod
    rows, c = W.phase1_lp(600, 800, 4)
    want = _infos(SimplexMethod(rows, c, engine="stream", max_pivots=12).get_solution())
    got = _infos(SimplexMethod(rows, c, engine="global", max_pivots=12).get_solution())
    assert len(got) == 14 and got[-1] == "pivot limit reached"
    assert got == want
    rows, c = W.phase1_lp(128, 256, 5)
    want = _infos(SimplexMethod(rows, c, engine="cluster", max_pivots=300).get_solution())
    got = _infos(SimplexMethod(rows, c, engine="global", max_pivots=300).get_solution())
    assert got == want
    with pytest.raises(ValueError, match="at most 14177 columns"):
        SimplexMethod(*W.dense_lp(1, 14178, 0), engine="global").get_solution()
