"""K7 (csrc/spx_cluster.cu): batches of mid-size LPs, one thread-block cluster per LP.

CPU part: the host-only capacity rule, argument validation and the cluster-size option (no device touched).
GPU part: bit-for-bit against the golden fixtures and the oracle at every cluster size, snapshots,
SimplexMethod(engine="cluster"), routing / launches and batch independence.
"""
import numpy as np
import pytest

import oracle
from simplex_method_solver_b200 import workloads as W
from util import END_TO_STATUS, bits, case_inputs, flat_of, label_codes, table_sha

OPT_CLUSTER_SIZE = 16
DYN_BYTES = 227 * 1024 - 2048
SIZES = (1, 2, 4, 8, 16)
# the shapes the GPU tests run, with the cluster size the library must pick for each
INTENDED_S = {(100, 100): 1, (128, 256): 2, (256, 300): 4, (3, 9000): 4, (256, 512): 8, (2000, 60): 8,
              (400, 800): 16, (512, 800): 16}


def footprint_fits(n, m, S):
    """Per-CTA shared memory of K7 (include/spx_b200.h, spx_solve_batched_cluster)."""
    R, Q = -(-n // S), -(-m // S)
    return 8 * (R * (m + 2) + 2 * m + 1) + 4 * (R + Q) <= DYN_BYTES


def expected_size(n, m):
    return next((S for S in SIZES if footprint_fits(n, m, S)), 0)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native.load()


class cluster_size:
    """Force SPX_OPT_CLUSTER_SIZE for the duration of a block (0 = automatic)."""

    def __init__(self, L, S):
        self.L, self.S = L, S

    def __enter__(self):
        assert self.L.spx_set_option(OPT_CLUSTER_SIZE, self.S) == 0

    def __exit__(self, *a):
        self.L.spx_set_option(OPT_CLUSTER_SIZE, 0)


# --------------------------------------------------------------------------- CPU
def test_cluster_size_follows_the_documented_footprint(lib):
    shapes = [(n, m) for n in (1, 2, 3, 17, 64, 100, 128, 255, 256, 400, 512, 528, 529, 1000, 2000, 5000)
              for m in (1, 2, 60, 100, 256, 300, 512, 800, 2000, 8000, 9499, 9500)]
    for n, m in shapes:
        assert lib.spx_cluster_size(n, m) == expected_size(n, m), (n, m)
    for (n, m), S in INTENDED_S.items():
        assert lib.spx_cluster_size(n, m) == S, (n, m)
    assert lib.spx_cluster_size(100, 100) == 1
    assert lib.spx_cluster_size(529, 800) == 0 and lib.spx_cluster_size(1, 9500) == 0
    assert lib.spx_cluster_size(528, 800) == 16 and lib.spx_cluster_size(1, 9499) == 16


def test_cluster_size_is_monotone(lib):
    for m in (1, 7, 100, 800, 4000):
        s = [lib.spx_cluster_size(n, m) for n in range(1, 700, 3)]
        nz = [v for v in s if v]
        assert nz == sorted(nz) and (0 not in s or all(v == 0 for v in s[s.index(0):])), m
    for n in (1, 10, 100, 400):
        s = [lib.spx_cluster_size(n, m) for m in range(1, 10000, 37)]
        nz = [v for v in s if v]
        assert nz == sorted(nz) and (0 not in s or all(v == 0 for v in s[s.index(0):])), n


def test_cluster_entry_validates_before_touching_the_device(lib):
    fake = 4096                                            # never dereferenced: validation fails first
    args = lambda T, B, n, m, rule, st, npv: (T, B, n, m, rule, 10, None, None, st, npv,  # noqa: E731
                                              None, None, None, None, None)
    for a, text in ((args(None, 1, 100, 100, 0, fake, fake), b"null"),
                    (args(fake, 1, 100, 100, 0, None, fake), b"null"),
                    (args(fake, 1, 100, 100, 0, fake, None), b"null"),
                    (args(fake, 1, 100, 100, 7, fake, fake), b"unknown rule"),
                    (args(fake, -1, 100, 100, 0, fake, fake), b"bad arguments"),
                    (args(fake, 1, 600, 800, 0, fake, fake), b"exceeds one cluster"),
                    (args(fake, 0, 1, 9500, 0, fake, fake), b"exceeds one cluster")):
        assert lib.spx_solve_batched_cluster(*a) < 0
        assert text in lib.spx_last_error(), (text, lib.spx_last_error())
    with cluster_size(lib, 1):                             # a forced size that does not fit is rejected
        assert lib.spx_solve_batched_cluster(*args(fake, 1, 128, 256, 0, fake, fake)) < 0
        assert b"SPX_OPT_CLUSTER_SIZE = 1" in lib.spx_last_error()
    assert lib.spx_solve_batched_cluster(*args(None, 0, 100, 100, 0, None, None)) == 0     # B = 0: nothing to do


def test_cluster_size_option_values(lib):
    try:
        assert lib.spx_get_option(OPT_CLUSTER_SIZE) == 0
        for v in (0, 1, 2, 4, 8, 16):
            assert lib.spx_set_option(OPT_CLUSTER_SIZE, v) == 0 and lib.spx_get_option(OPT_CLUSTER_SIZE) == v
        for v in (-1, 3, 5, 6, 12, 32):
            assert lib.spx_set_option(OPT_CLUSTER_SIZE, v) != 0
    finally:
        lib.spx_set_option(OPT_CLUSTER_SIZE, 0)
    assert lib.spx_get_option(OPT_CLUSTER_SIZE) == 0


def test_engine_routing_by_k4_footprint_needs_no_device(lib):
    from simplex_method_solver_b200.batched import kernel_for
    for n, m in ((8, 2), (4, 2), (20, 20), (64, 33), (99, 99), (1, 4469), (72, 136)):
        assert n * (m + 1) + m <= lib.spx_batched_max_cells()
        assert kernel_for(n, m) == "smem" and kernel_for(n, m, "smem") == "smem"
        assert kernel_for(n, m, "cluster") == "cluster"
    for n, m in ((1, 4470), (1, 4999), (2, 3228)):          # within 10,000 cells, but wider than one CTA holds
        assert n * (m + 1) + m <= lib.spx_batched_max_cells() and not lib.spx_batched_fits(n, m)
        assert kernel_for(n, m) == "cluster" and kernel_for(n, m, "auto_global") == "cluster"
        with pytest.raises(ValueError, match=f"a {n} x {m} LP .*does not fit the shared memory of one CTA"):
            kernel_for(n, m, "smem")
    for n, m in ((100, 100), (128, 256), (512, 800), (3, 9000)):
        assert kernel_for(n, m) == "cluster" and kernel_for(n, m, "cluster") == "cluster"
        with pytest.raises(ValueError):
            kernel_for(n, m, "smem")
    with pytest.raises(ValueError, match="at most n = 528 rows"):
        kernel_for(529, 800)
    with pytest.raises(ValueError, match="at most 9499 columns"):
        kernel_for(1, 9500, "cluster")
    with pytest.raises(ValueError, match="unknown engine"):
        kernel_for(8, 2, "warp")


# --------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def spx():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("GPU tests need a CUDA device")
    from simplex_method_solver_b200 import _native, batched, simplex

    class NS:
        pass
    ns = NS()
    ns.N, ns.L, ns.batched, ns.simplex, ns.torch = _native, _native.lib(), batched, simplex, torch
    return ns


def _check_golden(res, items, m):
    for k, (case, _) in enumerate(items):
        assert res.status[k] == END_TO_STATUS[case["end"]], case["name"]
        assert res.npiv[k] == len(case["trace"]), case["name"]
        assert res.trace[k, : res.npiv[k]].tolist() == case["trace"], case["name"]
        assert table_sha(res.tables[k]) == case["final_table_sha256"], case["name"]
        assert res.rowlab[k].tolist() == label_codes(case["row_labels"][:-1], m), case["name"]
        assert res.collab[k].tolist() == label_codes(case["column_labels"][:-1], m), case["name"]
        if "x1" in case:
            assert float(res.x[k, 0]).hex() == float(float.fromhex(case["x1"])).hex(), case["name"]
            assert float(res.x[k, 1]).hex() == float(float.fromhex(case["x2"])).hex(), case["name"]
            assert float(res.obj[k]).hex() == case["f"], case["name"]


def _groups(cases):
    groups = {}
    for case in cases:
        rows, c = case_inputs(case)
        groups.setdefault((rows.shape[0], rows.shape[1] - 1, case["cap"]), []).append((case, flat_of(rows, c)))
    return groups


@pytest.mark.gpu
@pytest.mark.parametrize("S", SIZES)
def test_all_reference_cases_through_the_cluster_solver(spx, ref_cases, dantzig_cases, S):
    """Every golden case, grouped by shape, at a forced cluster size (most have n < S: CTAs without rows)."""
    with cluster_size(spx.L, S):
        for (n, m, cap), items in _groups(ref_cases).items():
            assert footprint_fits(n, m, S)
            res = spx.batched.solve_batched(np.stack([f for _, f in items]), n, m, max_pivots=cap, engine="cluster")
            _check_golden(res, items, m)
        for (n, m, cap), items in _groups(dantzig_cases).items():
            if not footprint_fits(n, m, S):
                assert (n, m, S) == (40, 700, 1)           # 28,740 cells: two CTAs at least
                continue
            res = spx.batched.solve_batched(np.stack([f for _, f in items]), n, m, max_pivots=cap, rule="dantzig",
                                            engine="cluster")
            for k, (case, _) in enumerate(items):
                assert int(res.status[k]) == END_TO_STATUS[case["end"]], case["name"]
                assert res.trace[k, : int(res.npiv[k])].tolist() == case["trace"], case["name"]
                assert table_sha(res.tables[k]) == case["final_table_sha256"], case["name"]
                assert res.rowlab[k].tolist() == label_codes(case["row_labels"][:-1], m), case["name"]
                assert res.collab[k].tolist() == label_codes(case["column_labels"][:-1], m), case["name"]


def _family(kind, n, m, seed):
    if kind == "dense":
        return W.dense_lp(n, m, seed)
    if kind == "phase1":
        return W.phase1_lp(n, m, seed)
    rng = np.random.default_rng([seed, 7])
    rows, c = W.dense_lp(n, m, seed)
    if kind == "zeros":                                    # exact zeros: 0/p and zero-ratio paths
        rows[:, :m][rng.random((n, m)) < 0.3] = 0.0
        rows[rng.random(n) < 0.2, m] = 0.0
        return rows, c
    if kind == "incorrect":                                # a phase-1 row with no positive cell (:88-89)
        rows[n // 2, m] = -1.0
        return rows, c
    assert kind == "noconv"                                # the entering column has no eligible row (:138-139)
    rows[:, 0] = 0.0
    c[0] = -1.0
    return rows, c


def _check_oracle(res, flats, n, m, cap, rule="reference"):
    for k, T in enumerate(flats):
        o = oracle.solve_flat(T, n, m, max_pivots=cap, rule=rule)
        assert (int(res.status[k]), int(res.npiv[k])) == (o.status, o.npiv), (n, m, k)
        assert res.trace[k, : o.npiv].tolist() == o.trace.tolist(), (n, m, k)
        assert np.array_equal(bits(res.tables[k]), bits(o.table)), (n, m, k)
        assert res.rowlab[k].tolist() == o.rowlab.tolist() and res.collab[k].tolist() == o.collab.tolist()
        assert np.array_equal(bits(res.x[k]), bits(o.x)), (n, m, k)
        assert bits(res.obj[k]) == bits(o.obj2), (n, m, k)


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", sorted(INTENDED_S))
def test_mid_size_batches_against_the_oracle(spx, n, m):
    """One LP of each family per shape, every shape at its own cluster size (1, 2, 4, 8, 16)."""
    cap = 10_000
    assert spx.L.spx_cluster_size(n, m) == INTENDED_S[(n, m)]
    flats = [flat_of(*_family(kind, n, m, 100 + k))
             for k, kind in enumerate(("dense", "phase1", "zeros", "incorrect", "noconv"))]
    res = spx.batched.solve_batched(np.stack(flats), n, m, max_pivots=cap)
    _check_oracle(res, flats, n, m, cap)
    # a cap hit: half the oracle's pivot count on the first LP
    o = oracle.solve_flat(flats[0], n, m, max_pivots=cap)
    half = max(1, o.npiv // 2)
    res = spx.batched.solve_batched(flats[0][None, :], n, m, max_pivots=half)
    assert int(res.status[0]) == (oracle.CAP if o.npiv > half else o.status)
    _check_oracle(res, flats[:1], n, m, half)


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", [(128, 256), (2000, 60)])
def test_dantzig_rule_against_the_oracle(spx, n, m):
    flats = [flat_of(*_family(k, n, m, 5)) for k in ("dense", "phase1", "zeros")]
    res = spx.batched.solve_batched(np.stack(flats), n, m, max_pivots=10_000, rule="dantzig", engine="cluster")
    _check_oracle(res, flats, n, m, 10_000, rule="dantzig")


@pytest.mark.gpu
def test_snapshots_every_slot(spx):
    n, m, cap = 100, 100, 40
    flats = [flat_of(*W.phase1_lp(n, m, s)) for s in (1, 2, 3)]
    res = spx.batched.solve_batched(np.stack(flats), n, m, max_pivots=cap, snapshots=True)
    for k, T in enumerate(flats):
        o = oracle.solve_flat(T, n, m, max_pivots=cap, snapshots=True)
        assert int(res.npiv[k]) == o.npiv
        assert np.array_equal(bits(res.snaps[k, : o.npiv + 1]), bits(o.snaps))


@pytest.mark.gpu
def test_get_solution_on_the_cluster_engine(spx, ref_cases):
    from test_gpu_parity import _check_infos
    cases = [c for c in ref_cases if "get_solution" in c]
    assert len(cases) >= 15
    for case in cases:
        _check_infos(spx, case, "cluster")
    # a mid-size LP: every Info against the oracle's snapshots
    rows, c = W.phase1_lp(100, 100, 4)
    o = oracle.solve(rows, c, max_pivots=2000, snapshots=True)
    sm = spx.simplex.SimplexMethod(rows, c, engine="cluster")
    infos = sm.get_solution()
    assert len(infos) == o.npiv + 1 and o.status == oracle.OPTIMAL
    for q, info in enumerate(infos):
        flat = np.asarray([v for row in info.table for v in row])
        assert np.array_equal(bits(flat), bits(o.snaps[q])), q
        if q < o.npiv:
            assert (info.i, info.j) == tuple(o.trace[q])
    rl, cl = oracle.label_strings(o.rowlab, o.collab, 100)
    assert sm.row == rl and sm.column == cl
    # engine="auto" keeps its old route (streaming loop above 2048 cells)
    sm_auto = spx.simplex.SimplexMethod(rows, c)
    assert not sm_auto._use_warp()
    auto = sm_auto.get_solution()
    assert [(i.i, i.j) for i in auto] == [(i.i, i.j) for i in infos]


@pytest.mark.gpu
def test_routing_and_one_launch(spx):
    DB = spx.batched.DeviceBatch
    for n, m in ((8, 2), (20, 20), (64, 33), (99, 99)):
        assert DB(2, n, m).kernel == "smem"
    for n, m in ((100, 100), (128, 256), (3, 9000)):
        assert DB(2, n, m).kernel == "cluster"
    with pytest.raises(ValueError, match="capacity"):
        DB(2, 600, 800)
    T = np.stack([flat_of(*W.dense_lp(128, 256, s)) for s in range(3)])
    spx.L.spx_launch_count(1)
    spx.batched.solve_batched(T, 128, 256, max_pivots=50)
    assert spx.L.spx_launch_count(1) == 1
    spx.batched.solve_batched(flat_of(*W.dense_lp(20, 20, 1))[None, :], 20, 20, max_pivots=50)
    assert spx.L.spx_launch_count(1) == 1


@pytest.mark.gpu
def test_batch_independence(spx):
    n, m, cap = 100, 100, 10_000
    flats = np.stack([flat_of(*_family(("dense", "phase1", "zeros")[k % 3], n, m, 1000 + k)) for k in range(300)])
    full = spx.batched.solve_batched(flats, n, m, max_pivots=cap)
    o = oracle.solve_batched(flats, n, m, max_pivots=cap)
    assert np.array_equal(full.status, o.status) and np.array_equal(full.npiv, o.npiv)
    assert full.trace.tobytes() == o.trace.tobytes() and np.array_equal(bits(full.tables), bits(o.tables))
    assert np.array_equal(bits(full.x), bits(o.x)) and np.array_equal(bits(full.obj), bits(o.obj2))
    for k in (0, 1, 150, 299):
        one = spx.batched.solve_batched(flats[k][None, :], n, m, max_pivots=cap)
        for a, b in zip(one, full):
            if a is not None:
                assert a[0].tobytes() == b[k].tobytes(), k
    empty = spx.batched.solve_batched(flats[:0], n, m, max_pivots=cap)
    assert empty.status.shape == (0,) and empty.tables.shape == (0, n * (m + 1) + m)
