"""K8 (csrc/spx_global.cu): batches of LPs too large for one cluster's shared memory, one thread-block cluster per
LP with the table in global memory.

CPU part: the host-only capacity rule, argument validation, the cluster-size option and routing (no device touched).
GPU part: bit for bit against the golden fixtures at every cluster size, against the oracle above K7's capacity
and for a band above 2^24 cells, against K7 where both fit; snapshots, one launch per solve, batch independence,
the default cluster size.
"""
import numpy as np
import pytest

import oracle
from simplex_method_solver_b200 import workloads as W
from test_cluster_batched import _check_golden, _check_oracle, _family, _groups, cluster_size
from util import END_TO_STATUS, bits, flat_of, label_codes, table_sha

DYN_BYTES = 227 * 1024 - 2048
SIZES = (1, 2, 4, 8, 16)
INT32_MAX = (1 << 31) - 1
# shapes above K7's capacity: n just above its 528 rows at m = 800, tall, m above its 9,499 columns
LARGE = [(600, 800), (2000, 300), (64, 12000)]


def footprint_fits(n, m, S):
    """Per-CTA shared memory of K8 (include/spx_b200.h, spx_solve_batched_global)."""
    R, Q = -(-n // S), -(-m // S)
    return 8 * (2 * m + 1 + R) + 4 * (R + Q) <= DYN_BYTES


def expected_min_size(n, m):
    return next((S for S in SIZES if footprint_fits(n, m, S)), 0)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native.load()


def _args(T, B, n, m, rule, st, npv):
    return (T, B, n, m, rule, 10, None, None, st, npv, None, None, None, None, None)


# --------------------------------------------------------------------------- CPU
def test_min_cluster_size_follows_the_documented_footprint(lib):
    shapes = [(n, m) for n in (1, 2, 17, 100, 529, 600, 1000, 2000, 9000, 15866, 15867, 100000, 263856, 263857)
              for m in (1, 2, 300, 800, 2000, 9499, 9500, 10000, 11519, 11520, 12000, 14177, 14178)]
    for n, m in shapes:
        assert lib.spx_global_min_cluster_size(n, m) == expected_min_size(n, m), (n, m)
    assert lib.spx_global_min_cluster_size(0, 10) == 0 and lib.spx_global_min_cluster_size(10, 0) == 0


def test_capacity_edges(lib):
    smin = lib.spx_global_min_cluster_size
    # m at S = 1 and S = 16 (one row)
    assert smin(1, 11519) == 1 and smin(1, 11520) == 2
    assert smin(1, 14177) == 16 and smin(1, 14178) == 0
    assert footprint_fits(1, 11519, 1) and not footprint_fits(1, 11520, 1)
    assert footprint_fits(1, 14177, 16) and not footprint_fits(1, 14178, 16)
    # n at m = 800 / 2000 / 10000: the largest n at S = 1 and at S = 16
    for m in (800, 2000, 10000):
        for S in (1, 16):
            lo, hi = 1, 1 << 22
            while lo < hi:
                mid = (lo + hi + 1) // 2
                lo, hi = (mid, hi) if footprint_fits(mid, m, S) else (lo, mid - 1)
            if S == 1:
                assert smin(lo, m) == 1 and smin(lo + 1, m) > 1, (m, lo)
            else:
                assert smin(lo, m) == 16 and smin(lo + 1, m) == 0, (m, lo)
    assert smin(15866, 2000) == 1 and smin(15867, 2000) == 2
    assert smin(263856, 2000) == 16 and smin(263857, 2000) == 0


def test_global_entry_validates_before_touching_the_device(lib):
    fake = 4096                                            # never dereferenced: validation fails first
    for a, text in ((_args(None, 1, 600, 800, 0, fake, fake), b"null T/status/npiv"),
                    (_args(fake, 1, 600, 800, 0, None, fake), b"null T/status/npiv"),
                    (_args(fake, 1, 600, 800, 0, fake, None), b"null T/status/npiv"),
                    (_args(fake, 1, 600, 800, 7, fake, fake), b"unknown rule 7"),
                    (_args(fake, -1, 600, 800, 0, fake, fake), b"bad arguments"),
                    (_args(fake, 1, 0, 800, 0, fake, fake), b"bad arguments"),
                    (_args(fake, 1, 263857, 2000, 0, fake, fake), b"exceeds the shared memory of one cluster"),
                    (_args(fake, 0, 1, 14178, 0, fake, fake), b"230400 bytes"),
                    (_args(fake, INT32_MAX // 2 + 1, 1, 12000, 0, fake, fake), b"exceed one grid")):
        assert lib.spx_solve_batched_global(*a) < 0
        err = lib.spx_last_error()
        assert err.startswith(b"spx_solve_batched_global") and text in err, (text, err)
    with cluster_size(lib, 1):                             # a forced size that does not fit is rejected
        assert lib.spx_solve_batched_global(*_args(fake, 1, 1, 12000, 0, fake, fake)) < 0
        assert b"SPX_OPT_CLUSTER_SIZE = 1" in lib.spx_last_error()
        assert lib.spx_global_cluster_size(1, 12000, 1) == 0
    with cluster_size(lib, 16):                            # B * 16 CTAs beyond one grid
        assert lib.spx_solve_batched_global(*_args(fake, INT32_MAX // 16 + 1, 600, 800, 0, fake, fake)) < 0
        assert b"S = 16 CTAs exceed one grid" in lib.spx_last_error()
    assert lib.spx_solve_batched_global(*_args(None, 0, 600, 800, 0, None, None)) == 0      # B = 0: nothing to do


def test_forced_cluster_size_needs_no_device(lib):
    for S in SIZES:
        with cluster_size(lib, S):
            assert lib.spx_global_cluster_size(600, 800, 64) == S
            assert lib.spx_global_cluster_size(1, 12000, 1) == (S if S >= 2 else 0)


def test_engine_routing_needs_no_device(lib):
    from simplex_method_solver_b200.batched import ENGINES, kernel_for
    assert "global" in ENGINES
    for n, m in ((8, 2), (100, 100), (128, 256), (529, 800), (1000, 2000), (64, 12000), (9000, 2000)):
        assert kernel_for(n, m, "global") == "global"
    with pytest.raises(ValueError, match="at most n = 263856 rows"):
        kernel_for(263857, 2000, "global")
    with pytest.raises(ValueError, match="at most 14177 columns"):
        kernel_for(1, 14178, "global")
    # engine="auto" keeps every route: K4, K7, and an error above K7's capacity
    assert kernel_for(8, 2) == "smem" and kernel_for(128, 256) == "cluster"
    for n, m in ((529, 800), (1000, 2000), (9000, 2000)):
        with pytest.raises(ValueError, match="capacity"):
            kernel_for(n, m)
    with pytest.raises(ValueError, match="at most n = 528 rows"):
        kernel_for(529, 800)
    with pytest.raises(ValueError, match="at most 9499 columns"):
        kernel_for(64, 12000)


def test_sharded_batches_pass_the_engine_on():
    from simplex_method_solver_b200 import parallel as P
    seen = []

    def stand_in(tables, n, m, max_pivots, rule, device, engine="auto"):
        seen.append((tables.shape[0], n, m, engine))
        return "result"

    tabs = np.zeros((10, 600 * 801 + 800))
    start, count, res = P.solve_batched_sharded(tabs, 600, 800, max_pivots=5, rank=1, world=3, solver=stand_in,
                                                engine="global")
    assert (start, count, res) == (4, 3, "result") and seen == [(3, 600, 800, "global")]


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


def _solve(spx, flats, n, m, cap, **kw):
    return spx.batched.solve_batched(np.stack(flats), n, m, max_pivots=cap, engine="global", **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("S", SIZES)
def test_all_reference_cases_through_the_global_solver(spx, ref_cases, dantzig_cases, S):
    """Every golden case, grouped by shape, at a forced cluster size (most have n < S: CTAs without rows)."""
    with cluster_size(spx.L, S):
        for (n, m, cap), items in _groups(ref_cases).items():
            assert footprint_fits(n, m, S)
            res = _solve(spx, [f for _, f in items], n, m, cap)
            _check_golden(res, items, m)
        for (n, m, cap), items in _groups(dantzig_cases).items():
            assert footprint_fits(n, m, S)
            res = _solve(spx, [f for _, f in items], n, m, cap, rule="dantzig")
            for k, (case, _) in enumerate(items):
                assert int(res.status[k]) == END_TO_STATUS[case["end"]], case["name"]
                assert res.trace[k, : int(res.npiv[k])].tolist() == case["trace"], case["name"]
                assert table_sha(res.tables[k]) == case["final_table_sha256"], case["name"]
                assert res.rowlab[k].tolist() == label_codes(case["row_labels"][:-1], m), case["name"]
                assert res.collab[k].tolist() == label_codes(case["column_labels"][:-1], m), case["name"]


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", LARGE)
def test_large_batches_against_the_oracle(spx, n, m):
    """One LP of each family per shape above K7's capacity, at the default cluster size, and a cap hit."""
    cap = 10_000
    flats = [flat_of(*_family(kind, n, m, 100 + k))
             for k, kind in enumerate(("dense", "phase1", "zeros", "incorrect", "noconv"))]
    db = spx.batched.DeviceBatch(len(flats), n, m, max_pivots=cap, engine="global")
    assert db.kernel == "global" and db.cluster_size >= spx.L.spx_global_min_cluster_size(n, m)
    res = _solve(spx, flats, n, m, cap)
    _check_oracle(res, flats, n, m, cap)
    o = oracle.solve_flat(flats[0], n, m, max_pivots=cap)
    half = max(1, o.npiv // 2)
    res = _solve(spx, flats[:1], n, m, half)
    assert int(res.status[0]) == (oracle.CAP if o.npiv > half else o.status)
    _check_oracle(res, flats[:1], n, m, half)


@pytest.mark.gpu
def test_dantzig_rule_against_the_oracle(spx):
    n, m = 600, 800
    flats = [flat_of(*_family(k, n, m, 5)) for k in ("dense", "phase1", "zeros")]
    res = _solve(spx, flats, n, m, 10_000, rule="dantzig")
    _check_oracle(res, flats, n, m, 10_000, rule="dantzig")


@pytest.mark.gpu
def test_band_above_2_pow_24_cells(spx):
    """One CTA holding 18 M cells: the cell -> (row, column) map must stay exact."""
    n, m, cap = 9000, 2000, 30
    assert n * (m + 1) > 1 << 24
    T = flat_of(*W.phase1_lp(n, m, 3))
    with cluster_size(spx.L, 1):
        res = _solve(spx, [T], n, m, cap)
    o = oracle.solve_flat(T, n, m, max_pivots=cap)
    assert (int(res.status[0]), int(res.npiv[0])) == (o.status, o.npiv) and o.npiv == cap
    assert res.trace[0, :cap].tolist() == o.trace.tolist()
    got, want = res.tables[0], o.table
    body = n * (m + 1)
    assert np.array_equal(bits(got[body:]), bits(want[body:]))                        # f row
    assert np.array_equal(bits(got[m:body:m + 1]), bits(want[m:body:m + 1]))          # b column
    assert np.array_equal(bits(got), bits(want))                                      # the whole table
    assert np.array_equal(bits(res.x[0]), bits(o.x)) and res.collab[0].tolist() == o.collab.tolist()


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", [(128, 256), (400, 800)])
def test_same_bits_as_the_cluster_solver(spx, n, m):
    flats = [flat_of(*_family(kind, n, m, 7 + k)) for k, kind in enumerate(("dense", "phase1", "zeros"))]
    k7 = spx.batched.solve_batched(np.stack(flats), n, m, max_pivots=20_000, engine="cluster")
    k8 = _solve(spx, flats, n, m, 20_000)
    for a, b in zip(k7, k8):
        if a is not None:
            assert a.tobytes() == b.tobytes()


@pytest.mark.gpu
def test_snapshots_every_slot(spx):
    n, m, cap = 100, 100, 40
    flats = [flat_of(*W.phase1_lp(n, m, s)) for s in (1, 2, 3)]
    with cluster_size(spx.L, 4):
        res = _solve(spx, flats, n, m, cap, snapshots=True)
    for k, T in enumerate(flats):
        o = oracle.solve_flat(T, n, m, max_pivots=cap, snapshots=True)
        assert int(res.npiv[k]) == o.npiv
        assert np.array_equal(bits(res.snaps[k, : o.npiv + 1]), bits(o.snaps))


@pytest.mark.gpu
def test_one_launch_per_solve(spx):
    T = [flat_of(*W.dense_lp(600, 800, s)) for s in range(3)]
    spx.L.spx_launch_count(1)
    _solve(spx, T, 600, 800, 20)
    assert spx.L.spx_launch_count(1) == 1


@pytest.mark.gpu
def test_batch_independence_and_permutation(spx):
    n, m, cap = 200, 300, 10_000
    flats = np.stack([flat_of(*_family(("dense", "phase1", "zeros")[k % 3], n, m, 1000 + k)) for k in range(40)])
    full = _solve(spx, list(flats), n, m, cap)
    o = oracle.solve_batched(flats, n, m, max_pivots=cap)
    assert np.array_equal(full.status, o.status) and np.array_equal(full.npiv, o.npiv)
    assert np.array_equal(bits(full.tables), bits(o.tables)) and np.array_equal(bits(full.x), bits(o.x))
    perm = np.random.default_rng(1).permutation(len(flats))
    shuffled = _solve(spx, list(flats[perm]), n, m, cap)
    for a, b in zip(shuffled, full):
        if a is not None:
            assert a.tobytes() == b[perm].tobytes()
    for k in (0, 17, 39):
        one = _solve(spx, [flats[k]], n, m, cap)
        for a, b in zip(one, full):
            if a is not None:
                assert a[0].tobytes() == b[k].tobytes(), k
    empty = spx.batched.solve_batched(flats[:0], n, m, max_pivots=cap, engine="global")
    assert empty.status.shape == (0,) and empty.tables.shape == (0, n * (m + 1) + m)


@pytest.mark.gpu
def test_default_cluster_size(spx):
    for n, m in ((600, 800), (1000, 2000), (64, 12000)):
        smin = spx.L.spx_global_min_cluster_size(n, m)
        assert spx.L.spx_global_cluster_size(n, m, 1) == 16
        assert spx.L.spx_global_cluster_size(n, m, 10_000) == smin
        sizes = [spx.L.spx_global_cluster_size(n, m, B) for B in (1, 2, 4, 8, 16, 64, 256, 10_000)]
        assert sizes == sorted(sizes, reverse=True) and all(s >= smin for s in sizes)
