"""Every batched engine at the edges of its capacity, and every restatement of pick_element() on non-finite inputs.

CPU part: K4's capacity rule restated in Python (its CTA-mode footprint plus the kernel's 16 static bytes against
227 KB) over every shape of at most 10,000 cells, against spx_batched_fits, kernel_for, kernels_for and the ragged
plan under "auto" and "auto_global"; the adversarial-LP generator (each LP's decisive row is the one the oracle
picks), and the oracle against the original project on those LPs when $SIMPLEX_REF is set.
GPU part: LPs at the edge shapes of K4 (warp / CTA mode, each side of 48 KB, the last shapes one CTA holds), K7 (the
largest n at each cluster size) and K8 (the last columns one CTA holds, S = 16 full) through the uniform entries at
every cluster size that takes them, ragged batches, get_solution() and the sensitivity report, bit for bit against
the oracle; then the adversarial LPs (NaN, +-Inf, -0.0, subnormals, pivots of 2^+-300, overflow to Inf) with the
decisive row at the band edges of every cluster size, through every batched engine and every DeviceTableau loop.
"""
import hashlib

import numpy as np
import pytest

import oracle
from simplex_method_solver_b200 import workloads as W
from test_cluster_batched import _family, cluster_size, expected_size
from util import drive_reference, END_TO_STATUS, bits, flat_of

SIZES = (1, 2, 4, 8, 16)
KINDS = ("dense", "phase1", "zeros", "incorrect", "noconv")
MAX_CELLS = 10_000
K4_STATIC = 16                       # batched_kernel<true>'s s_ctl
K4_LIMIT = 227 * 1024 - K4_STATIC    # dynamic shared memory one K4 CTA may ask for
K8_BYTES = 227 * 1024 - 2048         # K7 and K8 per-CTA footprint limit (include/spx_b200.h)


def cells_of(n, m):
    return n * (m + 1) + m


def _ceil16(v):
    return (v + 15) // 16 * 16


def k4_footprint(n, m):
    """K4 CTA mode (csrc/spx_batched.cu): the cell -> (row, col) table, then two tables, x and the labels."""
    cells = cells_of(n, m)
    return _ceil16(4 * cells) + _ceil16(8 * (2 * cells + m) + 4 * (n + m))


def k4_fits(n, m):
    cells = cells_of(n, m)
    return cells <= MAX_CELLS and (cells <= 96 or k4_footprint(n, m) <= K4_LIMIT)


def k8_min_size(n, m):
    def fits(S):
        R, Q = -(-n // S), -(-m // S)
        return 8 * (2 * m + 1 + R) + 4 * (R + Q) <= K8_BYTES
    return next((S for S in SIZES if fits(S)), 0)


def triangle():
    """Every (n, m) with n, m >= 1 and at most 10,000 cells, as [k, 2] int64."""
    parts = []
    for n in range(1, (MAX_CELLS - 1) // 2 + 1):
        top = (MAX_CELLS - n) // (n + 1)
        parts.append(np.stack([np.full(top, n), np.arange(1, top + 1)], axis=1))
    return np.concatenate(parts).astype(np.int64)


def _shape(shapes, bad):
    return " x ".join(str(int(v)) for v in shapes[bad[0]])


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native.load()


# --------------------------------------------------------------------------- CPU: K4's capacity
def test_k4_routing_over_every_shape_of_at_most_10000_cells(lib):
    """"auto" and "auto_global" send an LP to K4 exactly when its CTA-mode footprint fits, and to K7 otherwise."""
    from simplex_method_solver_b200.batched import kernel_for, kernels_for, ragged_plan
    shapes = triangle()
    assert shapes.shape[0] == 73_671 and (cells_of(*shapes.T) <= MAX_CELLS).all()
    want = np.array([k4_fits(int(n), int(m)) for n, m in shapes])
    assert int((~want).sum()) == 635                                   # n = 1, m >= 4470 and n = 2, m >= 3228
    assert {(int(n), int(m)) for n, m in shapes[~want]} == (
        {(1, m) for m in range(4470, 5000)} | {(2, m) for m in range(3228, 3333)})
    for engine in ("auto", "auto_global"):
        got = np.array([kernel_for(int(n), int(m), engine) == "smem" for n, m in shapes])
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, f"kernel_for(..., {engine!r}): {bad.size} shapes, first {_shape(shapes, bad)}"
        kinds = np.array(kernels_for(shapes, engine))
        assert set(kinds[~want]) == {"cluster"} and set(kinds[want]) == {"smem"}, engine
        plan = ragged_plan(shapes, 0, engine)
        k4 = np.zeros(shapes.shape[0], dtype=bool)
        for la in plan.launches:
            k4[la["lps"]] = la["kind"] in ("warp", "cta")
            if la["kind"] == "cta":
                assert la["smem"] <= K4_LIMIT, engine
                assert la["smem"] == max(k4_footprint(*shapes[k]) for k in la["lps"]), engine
        bad = np.flatnonzero(k4 != want)
        assert bad.size == 0, f"ragged plan ({engine!r}): {bad.size} shapes, first {_shape(shapes, bad)}"


def test_k4_capacity_entry_and_smem_requests(lib):
    """spx_batched_fits is the same rule; engine="smem" still refuses a shape K4 cannot hold, naming the LP."""
    from simplex_method_solver_b200.batched import kernel_for, ragged_plan
    shapes = triangle()
    got = np.array([lib.spx_batched_fits(int(n), int(m)) for n, m in shapes])
    want = np.array([k4_fits(int(n), int(m)) for n, m in shapes])
    assert np.array_equal(got == 1, want) and set(got.tolist()) == {0, 1}
    for n, m in ((1, 5000), (72, 137), (100, 100), (0, 4), (4, 0), (-1, 3)):
        assert lib.spx_batched_fits(n, m) == 0
    for n, m in ((1, 4470), (1, 4999), (2, 3228), (2, 3332)):
        with pytest.raises(ValueError, match=rf"^a {n} x {m} LP \({cells_of(n, m)} cells\) does not fit"):
            kernel_for(n, m, "smem")
        with pytest.raises(ValueError, match=rf"LP 1: a {n} x {m} LP \({cells_of(n, m)} cells\) does not fit"):
            ragged_plan([(8, 2), (n, m)], 5, "smem")
    fake = 4096                                            # never dereferenced: validation fails first
    assert lib.spx_solve_batched(fake, 1, 1, 4470, 0, 10, None, None, fake, fake, None, None, None, None, None) < 0
    assert b"a 1 x 4470 LP (8941 cells) does not fit the shared memory of one CTA" in lib.spx_last_error()


# --------------------------------------------------------------------------- the edge shapes
def _k7_largest_n(m, S):
    """The largest n that K7 runs at cluster size S (spx_cluster_size(n, m) == S)."""
    n = 1
    while expected_size(n + 1, m) and expected_size(n + 1, m) <= S:
        n += 1
    return n


# (n, m) -> (kernel of "auto_global", its cluster size): "smem" (K4, S = 1), "cluster" (K7, spx_cluster_size),
# "global" (K8, S_min), None (refused by every engine).  No shape has 96 cells: (n+1)(m+1) = 97 is prime, so the
# largest warp-mode LPs have 95.
EDGES = {
    (11, 7): ("smem", 1), (7, 11): ("smem", 1), (13, 6): ("smem", 1),          # 95 / 95 / 97 cells: warp / CTA
    (1, 945): ("smem", 1), (96, 24): ("smem", 1),      # 49,168 B (above 48 KB) and exactly 49,152 B
    (50, 48): ("smem", 1), (72, 136): ("smem", 1),     # 72 x 136: 10,000 cells
    (1, 4469): ("smem", 1), (1, 4470): ("cluster", 1),  # the last width one CTA holds at n = 1 ...
    (2, 3227): ("smem", 1), (2, 3228): ("cluster", 1),  # ... and at n = 2
    (5, 1666): ("cluster", 1),                          # 10,001 cells
    **{(_k7_largest_n(m, S), m): ("cluster", S) for m in (800, 300) for S in SIZES},     # incl. 528 x 800
    (1, 9499): ("cluster", 16),
    (1, 11519): ("global", 1), (2, 11519): ("global", 2), (1, 11520): ("global", 2),
    (16, 14177): ("global", 16), (17, 14177): (None, 0),
}


def _cap(n, m):
    return 200 if cells_of(n, m) <= MAX_CELLS else 40


def test_edge_table_follows_the_footprints(lib):
    from simplex_method_solver_b200.batched import kernel_for
    assert _k7_largest_n(800, 16) == 528 and (528, 800) in EDGES
    for (n, m), (kind, S) in EDGES.items():
        if kind == "smem":
            assert k4_fits(n, m) and lib.spx_batched_fits(n, m) == 1 and kernel_for(n, m) == "smem", (n, m)
        elif kind == "cluster":
            assert not k4_fits(n, m) and lib.spx_cluster_size(n, m) == expected_size(n, m) == S, (n, m)
            assert kernel_for(n, m) == "cluster", (n, m)
            assert m not in (300, 800) or expected_size(n + 1, m) != S, (n, m)     # the largest n at S
        elif kind == "global":
            assert lib.spx_cluster_size(n, m) == 0 and lib.spx_global_min_cluster_size(n, m) == k8_min_size(n, m) == S
        else:
            assert lib.spx_global_min_cluster_size(n, m) == k8_min_size(n, m) == 0
            with pytest.raises(ValueError, match="capacity"):
                kernel_for(n, m, "auto_global")
        if kind is not None:
            assert kernel_for(n, m, "auto_global") == kind, (n, m)
    # the K8 footprint is exactly full at 16 x 14,177 (S = 16: R = 1, Q = 887) and 1 x 11,519 (S = 1)
    assert 8 * (2 * 14177 + 1 + 1) + 4 * (1 + 887) == K8_BYTES == 8 * (2 * 11519 + 1 + 1) + 4 * (1 + 11519)


def _route_grid():
    """The edge shapes, the K8 row limits at m = 2,000 (S = 1 and 16), and every shape one row or column away."""
    base = set(EDGES) | {(15866, 2000), (263856, 2000)}
    return sorted({(n + dn, m + dm) for n, m in base for dn in (-1, 0, 1) for dm in (-1, 0, 1) if n + dn and m + dm})


def test_route_agrees_with_kernel_for_the_plan_and_the_uniform_entries(lib):
    """spx_batched_route, kernel_for, the kind the ragged plan gives the LP and the uniform entry of that engine (B = 0,
    so nothing reaches the device) accept and refuse the same LPs, send them to the same kernel, and (without a forced
    cluster size) refuse with the same text; a forced size only adds the refusals of LPs that do not fit it."""
    from simplex_method_solver_b200 import _native as N
    from simplex_method_solver_b200.batched import ENGINE_CODES, kernel_for, ragged_plan
    from test_cluster_batched import footprint_fits
    entries = {"smem": lib.spx_solve_batched, "cluster": lib.spx_solve_batched_cluster,
               "global": lib.spx_solve_batched_global}
    kind_of = {N.ENGINE_SMEM: "smem", N.ENGINE_CLUSTER: "cluster", N.ENGINE_GLOBAL: "global"}
    plan_kind = {"warp": "smem", "cta": "smem", "cluster": "cluster", "global": "global"}
    routed = set()
    for forced in (0, 1, 16):
        with cluster_size(lib, forced):
            for n, m in _route_grid():
                for engine, code in ENGINE_CODES.items():
                    got = lib.spx_batched_route(n, m, code)
                    why = lib.spx_last_error().decode()
                    kind = kind_of.get(got)
                    assert (kind is None) == (got == -1), (n, m, engine, got)
                    if forced == 0:
                        routed.add((engine, kind))
                        try:
                            assert kernel_for(n, m, engine) == kind, (n, m, engine)
                        except ValueError as e:
                            assert kind is None and str(e) == why, (n, m, engine, str(e), why)
                    # a forced size refuses K7 and K8 LPs that do not fit it, and sets S
                    fits_forced = (forced == 0 or kind == "smem" or
                                   (kind == "cluster" and footprint_fits(n, m, forced)) or
                                   (kind == "global" and 0 < k8_min_size(n, m) <= forced))
                    accept = kind is not None and fits_forced
                    try:
                        plan = ragged_plan([(n, m)], 0, engine)
                        assert accept, (n, m, engine, forced)
                        (la,) = plan.launches
                        assert plan_kind[la["kind"]] == kind, (n, m, engine, forced)
                        if forced and kind != "smem":
                            assert la["S"] == forced
                        elif kind == "cluster":
                            assert la["S"] == expected_size(n, m)
                        elif kind == "global":
                            assert la["S"] == k8_min_size(n, m)
                    except ValueError as e:
                        assert not accept, (n, m, engine, forced, str(e))
                        assert forced or str(e) == f"spx_ragged_plan: LP 0: {why}", (str(e), why)
                    # the uniform entry of the engine the LP is routed to, or of the engine asked for
                    entry = entries[kind or engine] if engine in entries or kind else None
                    if entry is None:
                        continue
                    rc = entry(None, 0, n, m, 0, 10, None, None, None, None, None, None, None, None, None)
                    assert (rc == 0) == accept, (n, m, engine, forced, rc, lib.spx_last_error())
                    if rc != 0 and forced == 0:
                        assert lib.spx_last_error().decode() == f"{entry.__name__}: {why}"
    assert routed == {(e, k) for e in ENGINE_CODES for k in (None, "smem", "cluster", "global")} - {
        ("auto", "global"), ("smem", "cluster"), ("smem", "global"), ("cluster", "smem"), ("cluster", "global"),
        ("global", "smem"), ("global", "cluster")}


# --------------------------------------------------------------------------- the adversarial LPs
def band_rows(n):
    """Rows at band edges of every cluster size: k*R - 1 and k*R for the second and the last band (R = ceil(n/S))
    and n - 1."""
    rows = {n - 1}
    for S in SIZES:
        R = -(-n // S)
        for k in (1, -(-n // R) - 1):
            rows |= {k * R - 1, k * R}
    return sorted(r for r in rows if 0 <= r < n)


# (n, m): warp mode (83 cells), CTA mode; n is odd, so at S >= 2 the last band is short (or, at S = 16, empty)
SPECIAL_SHAPES = ((13, 5), (37, 6), (69, 6))
SPECIAL_KINDS = ("nan_first_col", "nan_first_b", "nan_later_col", "nan_later_b", "neg_inf", "tie_bands",
                 "zero_after_positive", "neg_zero_b", "neg_zero_col", "phase1_neg_inf", "f_neg_inf", "subnormal",
                 "pivot_2p300", "pivot_2m300", "overflow")
SPECIAL_CAP = 8


def adversarial(n, m, r0, kind, seed):
    """A dense LP (column 0 enters first: c[0] is the first negative cost) with one decisive value placed on row r0.
    Returns (rows, c, (row, col) the first pivot must be, or None where the kind does not fix it)."""
    inf, nan = float("inf"), float("nan")
    rows, c = W.dense_lp(n, m, seed)
    col, b = rows[:, 0], rows[:, m]                    # views
    expect = (r0, 0)
    if kind == "nan_first_col":                        # the first eligible ratio is NaN: that row wins (:117-121)
        col[:r0] = 0.0
        col[r0] = nan
    elif kind == "nan_first_b":
        col[:r0] = 0.0
        b[r0] = nan
    elif kind == "nan_later_col":                      # a later NaN ratio is never chosen
        col[r0] = nan
        expect = None
    elif kind == "nan_later_b":
        b[r0] = nan
        expect = None
    elif kind == "neg_inf":                            # every eligible ratio -Inf: the highest row (:133, '<=')
        col[r0 + 1:] = 0.0
        b[: r0 + 1] = inf
    elif kind == "tie_bands":                          # equal largest negative ratios in two bands: the higher row
        col[:] = -1.0
        b[:] = 10.0 + np.arange(n)
        p = 0 if r0 else n - 1
        b[r0] = b[p] = 1.0
        expect = (max(p, r0), 0)
    elif kind == "zero_after_positive":                # first eligible ratio positive, then zero ratios: first zero
        col[:] = 0.5
        b[r0] = 0.0
        b[n - 1] = 0.0
    elif kind == "neg_zero_b":                         # b = -0.0: a zero ratio, not a phase-1 row
        col[:] = 0.5
        b[r0] = -0.0
    elif kind == "neg_zero_col":                       # a = -0.0: not eligible (:112)
        col[:] = 0.5
        col[r0] = -0.0
        b[r0] = 1.0
        if r0 != n - 1:
            b[n - 1] = 0.0
            expect = (n - 1, 0)
        else:
            expect = None
    elif kind == "phase1_neg_inf":                     # phase-1 row with b = -Inf, +Inf its first positive cell
        rows[: r0, m] = np.abs(b[: r0])
        b[r0] = -inf
        rows[r0, :m] = -0.5
        rows[r0, m // 2] = inf
        expect = (r0, m // 2)
    elif kind == "f_neg_inf":                          # -Inf in the f row: entered by Dantzig, not by the reference
        c[0] = 0.5
        c[m - 1] = -inf
        rows[:, m - 1] = -1.0
        b[r0] = 0.5                                    # the largest negative ratio of column m - 1
        expect = None
    elif kind == "subnormal":                          # subnormal cells in the column, the pivot and elsewhere
        col[:] = -1e-320
        col[r0] = -1e-310
        b[r0] = 1e-310                                 # ratio -1, every other ratio -Inf or below -1e300
        rng = np.random.default_rng([seed, 3])
        body = rows[:, 1:m]
        body[rng.random(body.shape) < 0.3] = 4.9e-324
        c[1:][rng.random(m - 1) < 0.5] = -2.5e-310
    elif kind == "pivot_2p300":                        # pivots outside [2^-100, 2^100]: the fused update's fallback
        col[r0] = -(2.0 ** 300)
        b[r0] = 2.0 ** 299
    elif kind == "pivot_2m300":
        col[r0] = -(2.0 ** -300)
        b[r0] = 2.0 ** -301
    else:                                              # updates overflow to Inf; the next pivot meets Inf - Inf
        assert kind == "overflow", kind
        col[:] = 1e200
        col[r0] = -1.0
        b[r0] = 1.0
        rows[r0, 1:m:2] = -1e200
    return rows, c, expect


def special_lps(n, m):
    out = []
    for r0 in band_rows(n):
        for q, kind in enumerate(SPECIAL_KINDS):
            rows, c, expect = adversarial(n, m, r0, kind, seed=1000 * n + 50 * r0 + q)
            out.append((kind, r0, rows, c, expect))
    return out


def same(a, b):
    """Equal bits, or NaN on both sides (NaN payloads are not part of the contract)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))).all())


def test_band_rows_cover_every_band_edge():
    for n, _ in SPECIAL_SHAPES:
        rows = set(band_rows(n))
        assert n % 2 == 1 and n - 1 in rows
        for S in SIZES[1:]:
            R = -(-n // S)
            last = (n - 1) // R * R                      # first row of the last non-empty band
            assert n % S and {R - 1, R, last - 1, last} <= rows, (n, S)


def test_adversarial_lps_pivot_where_they_say():
    """The generator's decisive value decides the oracle's first pick, so the GPU tests exercise what they name."""
    seen = set()
    for n, m in SPECIAL_SHAPES:
        for kind, r0, rows, c, expect in special_lps(n, m):
            T = flat_of(rows, c)
            st, r, cc, _ = oracle.pick(T, n, m)
            if expect is not None:
                assert (st, r, cc) == (oracle.PIVOT, *expect), (n, m, kind, r0)
            if kind == "f_neg_inf":
                st, r, cc, _ = oracle.pick(T, n, m, rule="dantzig")
                assert (st, r, cc) == (oracle.PIVOT, r0, m - 1), (n, m, r0)
            o = oracle.solve_flat(T, n, m, max_pivots=SPECIAL_CAP)
            seen.add((kind, o.status))
            if kind == "overflow" and o.npiv >= 2:
                assert np.isinf(oracle.solve_flat(T, n, m, max_pivots=1).table).any()
                assert np.isnan(o.table).any(), (n, r0)                   # Inf - Inf on a later pivot
    assert {s for k, s in seen if k == "overflow"} & {oracle.CAP, oracle.OPTIMAL, oracle.NOCONV}
    assert len({k for k, _ in seen}) == len(SPECIAL_KINDS)


def test_oracle_against_the_reference_on_adversarial_lps(reference_module):
    """NaN / Inf behaviour of the oracle pinned to the original project, not only to itself."""
    if reference_module is None:
        pytest.skip("$SIMPLEX_REF is not set")
    for n, m in SPECIAL_SHAPES:
        for kind, r0, rows, c, _ in special_lps(n, m):
            end, trace, flat, _, _ = drive_reference(reference_module, rows, c, SPECIAL_CAP)
            o = oracle.solve_flat(flat_of(rows, c), n, m, max_pivots=SPECIAL_CAP)
            assert (END_TO_STATUS[end], trace) == (o.status, o.trace.tolist()), (n, kind, r0)
            assert same(flat, o.table), (n, kind, r0)


# --------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def spx():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("GPU tests need a CUDA device")
    from simplex_method_solver_b200 import _native, batched, engine, simplex

    class NS:
        pass
    ns = NS()
    ns.N, ns.L, ns.batched, ns.engine, ns.simplex, ns.torch = _native, _native.lib(), batched, engine, simplex, torch
    return ns


_ORACLE = {}


def oracle_of(T, n, m, cap, rule="reference"):
    key = (hashlib.sha1(T.tobytes()).digest(), n, m, cap, rule)
    if key not in _ORACLE:
        _ORACLE[key] = oracle.solve_flat(T, n, m, max_pivots=cap, rule=rule)
    return _ORACLE[key]


def check_one(one, k, T, n, m, cap, what, rule="reference"):
    """LP k of a BatchResult `one` against the oracle: status, npiv, trace, table, labels, x, obj (NaN == NaN)."""
    o = oracle_of(T, n, m, cap, rule)
    assert (int(one.status[k]), int(one.npiv[k])) == (o.status, o.npiv), (what, n, m, k)
    assert one.trace[k, : o.npiv].tolist() == o.trace.tolist(), (what, n, m, k)
    assert same(one.tables[k], o.table), (what, n, m, k)
    assert one.rowlab[k].tolist() == o.rowlab.tolist() and one.collab[k].tolist() == o.collab.tolist(), (what, k)
    assert same(one.x[k], o.x) and same(one.obj[k], o.obj2), (what, n, m, k)


def edge_batch(n, m):
    return [flat_of(*_family(kind, n, m, 7 * n + m + q)) for q, kind in enumerate(KINDS)]


def engine_runs(L, n, m, kind):
    """(engine, forced S or 0) of every uniform solve an n x m LP gets: "auto" ("auto_global" above K7), K7 at every
    S from its smallest to 16, K8 at its smallest S and at 16."""
    runs = [("auto_global" if kind == "global" else "auto", 0)]
    s7 = L.spx_cluster_size(n, m)
    runs += [("cluster", S) for S in SIZES if s7 and S >= s7]
    s8 = L.spx_global_min_cluster_size(n, m)
    runs += [("global", S) for S in sorted({s8, 16}) if s8]
    return runs


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", sorted(EDGES))
def test_edge_shape_every_engine_against_the_oracle(spx, n, m):
    kind, S_want = EDGES[(n, m)]
    B = spx.batched
    if kind is None:
        for engine in ("auto", "auto_global", "cluster", "global"):
            with pytest.raises(ValueError, match="capacity"):
                B.DeviceBatch(1, n, m, engine=engine)
        return
    db = B.DeviceBatch(5, n, m, engine="auto_global")
    assert db.kernel == kind
    if kind == "cluster":
        assert spx.L.spx_cluster_size(n, m) == S_want
    if kind == "global":
        assert spx.L.spx_global_min_cluster_size(n, m) == S_want
    flats = np.stack(edge_batch(n, m))
    cap = _cap(n, m)
    first = None
    for engine, S in engine_runs(spx.L, n, m, kind):
        with cluster_size(spx.L, S):
            res = B.solve_batched(flats, n, m, max_pivots=cap, engine=engine)
        for k in range(flats.shape[0]):
            check_one(res, k, flats[k], n, m, cap, (engine, S))
        first = first or res
    ends = {int(s) for s in first.status}
    assert oracle.INCORRECT in ends and oracle.NOCONV in ends, ends
    # the sensitivity report of the optimal LPs against the sequential statement
    import sensitivity_oracle as SO
    rep = B.sensitivity(first)
    for k in np.flatnonzero(first.status == oracle.OPTIMAL):
        want = SO.sensitivity(first.tables[k], n, m, first.rowlab[k], first.collab[k], True)
        for g, w in zip(rep[:5], want):
            assert same(g[k], w), (n, m, k)
    assert rep.optimal.tolist() == (first.status == oracle.OPTIMAL).tolist()


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", sorted(nm for nm, (kind, _) in EDGES.items() if cells_of(*nm) <= MAX_CELLS))
def test_get_solution_warp_engine_at_the_k4_edges(spx, n, m):
    rows, c = W.phase1_lp(n, m, n + m)
    if not k4_fits(n, m):
        with pytest.raises(ValueError, match="engine='warp'"):
            spx.simplex.SimplexMethod(rows, c, engine="warp").get_solution()
        return
    cap = 100
    o = oracle.solve(rows, c, max_pivots=cap, snapshots=True)
    infos = spx.simplex.SimplexMethod(rows, c, engine="warp", max_pivots=cap).get_solution()
    tables = [i for i in infos if isinstance(i, spx.simplex.Info)]
    assert len(tables) == o.npiv + 1
    for q, info in enumerate(tables):
        assert np.array_equal(bits(np.asarray([v for row in info.table for v in row])), bits(o.snaps[q])), q
        if q < o.npiv:
            assert (info.i, info.j) == tuple(o.trace[q]), q
    assert isinstance(infos[-1], spx.simplex.Error) == (o.status != oracle.OPTIMAL)


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["auto", "auto_global", "global"])
def test_edge_shapes_in_one_ragged_batch(spx, engine):
    from simplex_method_solver_b200.batched import kernel_for
    lps, shapes = [], []
    for (n, m), (kind, _) in sorted(EDGES.items()):
        if kind is None or (engine == "auto" and kind == "global"):
            continue
        for T in edge_batch(n, m):
            lps.append((T[: n * (m + 1)].reshape(n, m + 1), T[n * (m + 1):]))
            shapes.append((n, m))
    caps = [_cap(n, m) for n, m in shapes]
    res = spx.batched.solve_ragged(lps, max_pivots=caps, engine=engine)
    for k, (n, m) in enumerate(shapes):
        if engine != "global":
            assert kernel_for(n, m, engine) == EDGES[(n, m)][0]
        check_one(res.lp(k), 0, flat_of(*lps[k]), n, m, caps[k], ("ragged", engine))


SPECIAL_RUNS = [("auto", 0)] + [("cluster", S) for S in SIZES] + [("global", S) for S in SIZES]


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["reference", "dantzig"])
def test_special_values_every_batched_engine(spx, rule):
    """The adversarial LPs through K4 (warp and CTA mode), K7 and K8 at every cluster size, uniform and ragged."""
    B = spx.batched
    every = []
    for n, m in SPECIAL_SHAPES:
        lps = special_lps(n, m)
        flats = np.stack([flat_of(rows, c) for _, _, rows, c, _ in lps])
        every += [(n, m, rows, c) for _, _, rows, c, _ in lps]
        for engine, S in SPECIAL_RUNS:
            with cluster_size(spx.L, S):
                res = B.solve_batched(flats, n, m, max_pivots=SPECIAL_CAP, rule=rule, engine=engine)
            for k, (kind, r0, *_rest) in enumerate(lps):
                check_one(res, k, flats[k], n, m, SPECIAL_CAP, (engine, S, kind, r0), rule)
    lps = [(rows, c) for _, _, rows, c in every]
    for engine, S in [("auto_global", 0)] + SPECIAL_RUNS:
        with cluster_size(spx.L, S):
            res = B.solve_ragged(lps, max_pivots=SPECIAL_CAP, rule=rule, engine=engine)
        for k, (n, m, rows, c) in enumerate(every):
            check_one(res.lp(k), 0, flat_of(rows, c), n, m, SPECIAL_CAP, ("ragged", engine, S), rule)


LOOPS = [False, True, "resident", "fused", "fused-coop", "fused-gpuwide", "fused-engine"]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", LOOPS)
def test_special_values_every_device_tableau_loop(spx, mode):
    """The adversarial LPs through the pivot-at-a-time, look-ahead, L2-resident and fused loops of spx_solve."""
    from test_gpu_parity import loop_mode
    N = spx.N
    for n, m in SPECIAL_SHAPES:
        dev = spx.engine.DeviceTableau(n, m, trace_capacity=SPECIAL_CAP)
        for kind, r0, rows, c, _ in special_lps(n, m):
            for rule in (("reference", "dantzig") if kind == "f_neg_inf" else ("reference",)):
                o = oracle_of(flat_of(rows, c), n, m, SPECIAL_CAP, rule)
                dev.load(np.ascontiguousarray(rows), np.ascontiguousarray(c), max_pivots=SPECIAL_CAP)
                with loop_mode(mode) as mode_:
                    status, npiv = dev.solve(rule=N.RULES[rule], lookahead=mode_)
                what = (mode, rule, n, kind, r0)
                assert (status, npiv) == (o.status, o.npiv), what
                assert dev.trace[:npiv].cpu().numpy().tolist() == o.trace.tolist(), what
                assert same(dev.export_flat(npiv), o.table), what
                rl, cl = dev.labels_host()
                assert rl.tolist() == o.rowlab.tolist() and cl.tolist() == o.collab.tolist(), what
