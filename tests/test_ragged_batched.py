"""Ragged batches: LPs of any mix of shapes in one call (spx_ragged_plan + spx_solve_batched_ragged, batched.solve_ragged).

CPU part: the host-only plan (offsets, routing, launch order and count, validation), the solve entry's checks before the
device is touched, and the cell-balanced split of parallel.solve_ragged_sharded.
GPU part: the golden sets in one call each, every forced cluster size, a mixed batch of the five families against the
oracle, snapshots, independence from the batch and its order, launch counts, reuse, the empty batch, multi-GPU.
"""
import os
import socket
import sys

import numpy as np
import pytest

import oracle
from simplex_method_solver_b200 import workloads as W
from test_cluster_batched import _family, cluster_size
from util import END_TO_STATUS, bits, case_inputs, flat_of, label_codes, table_sha

SIZES = (1, 2, 4, 8, 16)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native.load()


def cells_of(n, m):
    return n * (m + 1) + m


def expected_class(L, n, m, engine="auto"):
    """("warp" | "cta" | "cluster", S) of an LP, from the uniform entries' own rules."""
    from simplex_method_solver_b200.batched import kernel_for
    if kernel_for(n, m, engine) == "smem":
        return ("warp" if cells_of(n, m) <= 96 else "cta"), 1
    forced = L.spx_get_option(16)
    return "cluster", (forced or L.spx_cluster_size(n, m))


def expected_launches(L, shapes, engine="auto"):
    return len({expected_class(L, n, m, engine) for n, m in shapes})


def random_shapes(rng, B):
    """Shapes across warp mode, CTA mode and every cluster size."""
    out = []
    for _ in range(B):
        kind = rng.integers(0, 3)
        if kind == 0:
            out.append((int(rng.integers(1, 12)), int(rng.integers(1, 7))))
        elif kind == 1:
            out.append((int(rng.integers(5, 99)), int(rng.integers(5, 99))))
        else:
            out.append((int(rng.integers(60, 528)), int(rng.integers(100, 801))))
    return out


# --------------------------------------------------------------------------- CPU
def test_plan_offsets_are_prefix_sums(lib):
    from simplex_method_solver_b200.batched import ragged_plan
    rng = np.random.default_rng(1)
    for B in (1, 2, 7, 300):
        shapes = random_shapes(rng, B)
        caps = rng.integers(0, 300, B)
        p = ragged_plan(shapes, caps)
        n, m = np.array(shapes).T
        cells = n * (m + 1) + m
        excl = lambda v: np.concatenate([[0], np.cumsum(v)[:-1]])  # noqa: E731
        assert p.lps["n"].tolist() == n.tolist() and p.lps["m"].tolist() == m.tolist()
        assert p.lps["max_pivots"].tolist() == caps.tolist() and p.lps["cells"].tolist() == cells.tolist()
        for field, v in (("t", cells), ("xm", m), ("xn", n), ("tr", caps), ("sn", (caps + 1) * cells)):
            assert p.lps[field].tolist() == excl(v).tolist(), field
        assert p.totals.tolist() == [cells.sum(), m.sum(), n.sum(), caps.sum(), ((caps + 1) * cells).sum()]


@pytest.mark.parametrize("engine", ["auto", "smem", "cluster"])
def test_plan_routing_order_and_launch_count(lib, engine):
    from simplex_method_solver_b200.batched import kernels_for, ragged_plan
    rng = np.random.default_rng(2)
    shapes = random_shapes(rng, 400)
    if engine == "smem":
        shapes = [(n, m) for n, m in shapes if cells_of(n, m) <= 5000]
    shapes += shapes[:5]                                   # equal cells: ties by index
    p = ragged_plan(shapes, 10, engine)
    seen = []
    for la in p.launches:
        idx = la["lps"].tolist()
        seen += idx
        for k in idx:
            assert expected_class(lib, *shapes[k], engine) == (la["kind"], la["S"]), (k, shapes[k])
        key = [(-cells_of(*shapes[k]), k) for k in idx]
        assert key == sorted(key), "largest first, ties by batch index"
    assert sorted(seen) == list(range(len(shapes)))
    assert len(p.launches) == expected_launches(lib, shapes, engine)
    kinds = kernels_for(shapes, engine)
    assert kinds == [("cluster" if expected_class(lib, n, m, engine)[0] == "cluster" else "smem") for n, m in shapes]


def test_plan_at_every_forced_cluster_size(lib):
    from simplex_method_solver_b200.batched import ragged_plan
    shapes = [(100, 100), (128, 256), (40, 700), (300, 200), (8, 2)]
    for S in SIZES:
        with cluster_size(lib, S):
            fits = [(n, m) for n, m in shapes if cells_of(n, m) <= 96 or
                    lib.spx_cluster_size(n, m) and lib.spx_cluster_size(n, m) <= S]
            p = ragged_plan(fits, 10, "cluster")
            assert {la["S"] for la in p.launches} == {S} and len(p.launches) == 1


def test_launch_count_formula_cases(lib):
    from simplex_method_solver_b200.batched import ragged_plan
    for shapes, count in (([(8, 2)], 1), ([(8, 2), (20, 20)], 2), ([(100, 100), (128, 256)], 2),
                          ([(8, 2), (20, 20), (100, 100), (128, 256), (256, 300), (256, 512), (400, 800)], 7),
                          ([(3, 2)] * 5 + [(512, 800)], 2)):
        assert len(ragged_plan(shapes, 5).launches) == count == expected_launches(lib, shapes)


def _plan_raw(L, shapes, engine=0, nbytes=None):
    import ctypes
    h = np.ascontiguousarray(np.asarray(shapes, dtype=np.int32).reshape(-1, 3))
    B = h.shape[0]
    need = L.spx_ragged_plan_bytes(B)
    buf = np.zeros(max(need, 16), dtype=np.uint8)
    tot = np.zeros(5, dtype=np.int64)
    rc = L.spx_ragged_plan(h.ctypes.data, B, engine, buf.ctypes.data, need if nbytes is None else nbytes,
                           tot.ctypes.data)
    return rc, ctypes.string_at(L.spx_last_error()), buf


def test_plan_validation_names_the_lp_and_sends_wide_k4_shapes_to_k7(lib):
    for bad, text in (([(4, 2, 10), (0, 2, 10)], b"LP 1: bad shape n=0"),
                      ([(4, 2, 10), (4, 2, 10), (4, 0, 10)], b"LP 2: bad shape n=4 m=0"),
                      ([(4, 2, -1)], b"LP 0: bad shape n=4 m=2 max_pivots=-1"),
                      ([(4, 2, 5), (100, 100, 5), (529, 800, 5), (8, 2, 5)], b"LP 2: a 529 x 800 LP exceeds one cluster")):
        rc, err, _ = _plan_raw(lib, bad)
        assert rc < 0 and text in err, err
    rc, err, _ = _plan_raw(lib, [(4, 2, 5), (529, 800, 5)])
    assert b"230400 bytes" in err                          # the capacity
    rc, err, _ = _plan_raw(lib, [(8, 2, 5), (100, 100, 5)], engine=1)
    assert rc < 0 and b"LP 1: 10200 cells per LP exceed the shared-memory resident limit 10000" in err, err
    with cluster_size(lib, 1):
        rc, err, _ = _plan_raw(lib, [(100, 100, 5), (128, 256, 5)])
        assert rc < 0 and b"LP 1: a 128 x 256 LP does not fit a cluster of SPX_OPT_CLUSTER_SIZE = 1 CTAs" in err, err
    rc, err, _ = _plan_raw(lib, [(8, 2, 5), (1, 4999, 5)], engine=1)   # 9,999 cells, 260 KB: K4 cannot hold it
    assert rc < 0 and b"LP 1: a 1 x 4999 LP (9999 cells) does not fit the shared memory of one CTA" in err, err
    rc, err, _ = _plan_raw(lib, [(8, 2, 5), (1, 4999, 5)])              # "auto" gives it to K7
    assert rc == 0, err
    rc, err, _ = _plan_raw(lib, [(8, 2, 5)] * 3, nbytes=lib.spx_ragged_plan_bytes(3) - 1)
    assert rc < 0 and b"plan_bytes" in err
    rc, err, _ = _plan_raw(lib, [(8, 2, 5)], engine=3)
    assert rc < 0 and b"unknown engine" in err
    assert lib.spx_ragged_plan_bytes(-1) == -1


def test_python_routing_names_the_lp(lib):
    from simplex_method_solver_b200.batched import kernels_for, ragged_plan, _caps
    with pytest.raises(ValueError, match=r"^LP 2: a 529 x 800 LP .*at most n = 528 rows"):
        kernels_for([(8, 2), (100, 100), (529, 800), (600, 800)])
    with pytest.raises(ValueError, match=r"^LP 1: 10200 cells per LP exceed"):
        kernels_for([(8, 2), (100, 100)], "smem")
    with pytest.raises(ValueError, match=r"^LP 1: max_pivots = -1"):
        _caps([3, -1], 2)
    with pytest.raises(ValueError, match="one int per LP"):
        _caps([3, 4, 5], 2)
    with pytest.raises(ValueError, match="LP 1: bad shape"):
        ragged_plan([(8, 2), (0, 2)], 5)


def test_solve_entry_validates_before_touching_the_device(lib):
    fake = 4096                                            # never dereferenced: validation fails first
    rc, _, plan = _plan_raw(lib, [(8, 2, 5), (100, 100, 5)])
    assert rc == 0

    def solve(h_plan, d_plan=fake, T=fake, rule=0, st=fake, npv=fake):
        return lib.spx_solve_batched_ragged(T, h_plan, d_plan, rule, None, None, st, npv, None, None, None, None, None)

    for kw, text in (({"h_plan": None}, b"null plan"), ({"h_plan": plan.ctypes.data, "d_plan": None}, b"null"),
                     ({"h_plan": plan.ctypes.data, "T": None}, b"null"),
                     ({"h_plan": plan.ctypes.data, "st": None}, b"null"),
                     ({"h_plan": plan.ctypes.data, "npv": None}, b"null"),
                     ({"h_plan": plan.ctypes.data, "rule": 7}, b"unknown rule")):
        assert solve(**kw) < 0
        assert text in lib.spx_last_error(), (kw, lib.spx_last_error())
    bad = plan.copy()
    bad[:4] = 0                                            # magic
    assert solve(bad.ctypes.data) < 0 and b"magic" in lib.spx_last_error()
    bad = plan.copy()
    bad[4:8] = np.frombuffer(np.int32(5).tobytes(), np.uint8)    # ABI version
    assert solve(bad.ctypes.data) < 0 and b"ABI version" in lib.spx_last_error()
    bad = plan.copy()
    bad[8:16] = np.frombuffer(np.int64(3).tobytes(), np.uint8)   # B no longer matches the launches
    assert solve(bad.ctypes.data) < 0 and b"inconsistent plan" in lib.spx_last_error()
    rc, _, empty = _plan_raw(lib, np.zeros((0, 3)))
    assert rc == 0
    assert solve(empty.ctypes.data, d_plan=None, T=None, st=None, npv=None) == 0      # B = 0: nothing to do


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_solve_ragged_sharded_balances_cells(world):
    from simplex_method_solver_b200.parallel import solve_ragged_sharded
    rng = np.random.default_rng(world)
    lps = [W.dense_lp(int(rng.integers(1, 60)), int(rng.integers(2, 200)), s) for s in range(97)]
    lps += [W.dense_lp(400, 700, 1)] + [W.dense_lp(2, 3, s) for s in range(20)]
    cells = np.array([r.size + c.size for r, c in lps])
    caps = list(range(len(lps)))
    calls = []

    def stand_in(part, max_pivots, rule, trace, snapshots, device, engine):
        calls.append((len(part), list(max_pivots), rule, engine))
        return "result"

    got = []
    for rank in range(world):
        start, count, res = solve_ragged_sharded(lps, max_pivots=caps, rule="dantzig", rank=rank, world=world,
                                                 solver=stand_in, engine="cluster")
        assert res == "result" and calls[-1] == (count, caps[start:start + count], "dantzig", "cluster")
        assert cells[start:start + count].sum() <= cells.sum() / world + cells.max()
        got.append((start, count))
    assert got[0][0] == 0 and sum(c for _, c in got) == len(lps)
    for (s0, c0), (s1, _) in zip(got, got[1:]):
        assert s0 + c0 == s1


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


def _check_case(one, case, m):
    """one: res.lp(k); as test_cluster_batched._check_golden for one case."""
    name = case["name"]
    assert int(one.status[0]) == END_TO_STATUS[case["end"]], name
    assert int(one.npiv[0]) == len(case["trace"]), name
    assert one.trace[0, : int(one.npiv[0])].tolist() == case["trace"], name
    assert table_sha(one.tables[0]) == case["final_table_sha256"], name
    assert one.rowlab[0].tolist() == label_codes(case["row_labels"][:-1], m), name
    assert one.collab[0].tolist() == label_codes(case["column_labels"][:-1], m), name
    if "x1" in case:
        assert float(one.x[0, 0]).hex() == float(float.fromhex(case["x1"])).hex(), name
        assert float(one.x[0, 1]).hex() == float(float.fromhex(case["x2"])).hex(), name
        assert float(one.obj[0]).hex() == case["f"], name


def _golden_lps(cases):
    lps = [case_inputs(c) for c in cases]
    return lps, [c["cap"] for c in cases]


@pytest.mark.gpu
def test_all_reference_cases_in_one_call(spx, ref_cases):
    lps, caps = _golden_lps(ref_cases)
    assert len(ref_cases) == 381 and set(caps) == {25, 200, 5000}
    spx.L.spx_launch_count(1)
    res = spx.batched.solve_ragged(lps, max_pivots=caps)
    assert spx.L.spx_launch_count(1) == expected_launches(spx.L, [(r.shape[0], c.shape[0]) for r, c in lps])
    for k, case in enumerate(ref_cases):
        _check_case(res.lp(k), case, lps[k][1].shape[0])


@pytest.mark.gpu
def test_all_dantzig_cases_in_one_call(spx, dantzig_cases):
    lps, caps = _golden_lps(dantzig_cases)
    assert len(dantzig_cases) == 154
    db = spx.batched.DeviceRaggedBatch([(r.shape[0], c.shape[0]) for r, c in lps], caps)
    big = [k for k, (r, c) in enumerate(lps) if (r.shape[0], c.shape[0]) == (40, 700)]
    assert big and all(db.kernels[k] == "cluster" for k in big)
    assert all(db.kernels[k] == "smem" for k in range(len(lps)) if k not in big)
    res = spx.batched.solve_ragged(lps, max_pivots=caps, rule="dantzig")
    for k, case in enumerate(dantzig_cases):
        one, m = res.lp(k), lps[k][1].shape[0]
        assert int(one.status[0]) == END_TO_STATUS[case["end"]], case["name"]
        assert one.trace[0, : int(one.npiv[0])].tolist() == case["trace"], case["name"]
        assert table_sha(one.tables[0]) == case["final_table_sha256"], case["name"]
        assert one.rowlab[0].tolist() == label_codes(case["row_labels"][:-1], m), case["name"]
        assert one.collab[0].tolist() == label_codes(case["column_labels"][:-1], m), case["name"]


@pytest.mark.gpu
@pytest.mark.parametrize("S", SIZES)
def test_reference_cases_at_every_forced_cluster_size(spx, ref_cases, S):
    lps, caps = _golden_lps(ref_cases)
    with cluster_size(spx.L, S):
        db = spx.batched.DeviceRaggedBatch([(r.shape[0], c.shape[0]) for r, c in lps], caps, engine="cluster")
        assert db.launches == 1 and set(db.kernels) == {"cluster"}
        res = spx.batched.solve_ragged(lps, max_pivots=caps, engine="cluster")
    for k, case in enumerate(ref_cases):
        _check_case(res.lp(k), case, lps[k][1].shape[0])


MIXED_SHAPES = [(4, 2), (8, 2), (3, 5), (11, 6), (12, 20), (30, 30), (64, 33), (99, 99), (1, 3000),
                (100, 100), (128, 256), (256, 300), (256, 512), (400, 800), (3, 9000)]


def _mixed(count, seed, cap_max=3000):
    """~count LPs of the five families over MIXED_SHAPES (warp mode, CTA mode, S = 1, 2, 4, 8, 16), caps incl. 0."""
    rng = np.random.default_rng(seed)
    kinds = ("dense", "phase1", "zeros", "incorrect", "noconv")
    lps, caps = [], []
    for q in range(count):
        n, m = MIXED_SHAPES[q % len(MIXED_SHAPES)]
        lps.append(_family(kinds[(q // len(MIXED_SHAPES)) % 5], n, m, 300 + q))
        caps.append(0 if q % 23 == 5 else int(rng.integers(1, cap_max)))
    return lps, caps


@pytest.mark.gpu
def test_mixed_batch_against_the_oracle(spx):
    lps, caps = _mixed(200, 1)
    classes = {expected_class(spx.L, n, m) for n, m in MIXED_SHAPES}
    assert classes == {("warp", 1), ("cta", 1)} | {("cluster", S) for S in SIZES}
    spx.L.spx_launch_count(1)
    res = spx.batched.solve_ragged(lps, max_pivots=caps)
    assert spx.L.spx_launch_count(1) == 7
    ends = set()
    for k, (rows, c) in enumerate(lps):
        n, m = rows.shape[0], c.shape[0]
        o = oracle.solve_flat(flat_of(rows, c), n, m, max_pivots=caps[k])
        one = res.lp(k)
        ends.add(o.status)
        assert (int(one.status[0]), int(one.npiv[0])) == (o.status, o.npiv), (k, n, m)
        assert one.trace[0, : o.npiv].tolist() == o.trace.tolist(), k
        assert np.array_equal(bits(one.tables[0]), bits(o.table)), k
        assert one.rowlab[0].tolist() == o.rowlab.tolist() and one.collab[0].tolist() == o.collab.tolist(), k
        assert np.array_equal(bits(one.x[0]), bits(o.x)) and bits(one.obj[0]) == bits(o.obj2), k
    assert {oracle.CAP, oracle.OPTIMAL, oracle.INCORRECT, oracle.NOCONV} <= ends


@pytest.mark.gpu
def test_snapshots_every_slot(spx):
    shapes = [(4, 2), (12, 20), (100, 100), (128, 256), (8, 2), (30, 30)]
    lps = [W.phase1_lp(n, m, s) for s, (n, m) in enumerate(shapes)]
    caps = [6, 25, 30, 12, 0, 40]
    res = spx.batched.solve_ragged(lps, max_pivots=caps, snapshots=True)
    for k, (rows, c) in enumerate(lps):
        n, m = rows.shape[0], c.shape[0]
        o = oracle.solve_flat(flat_of(rows, c), n, m, max_pivots=caps[k], snapshots=True)
        one = res.lp(k)
        assert int(one.npiv[0]) == o.npiv and one.snaps.shape == (1, caps[k] + 1, cells_of(n, m))
        assert np.array_equal(bits(one.snaps[0, : o.npiv + 1]), bits(o.snaps)), k


@pytest.mark.gpu
def test_independence_and_order(spx):
    lps, caps = _mixed(60, 2, cap_max=800)
    res = spx.batched.solve_ragged(lps, max_pivots=caps)
    for k, (rows, c) in enumerate(lps):
        n, m = rows.shape[0], c.shape[0]
        alone = spx.batched.solve_batched(flat_of(rows, c)[None, :], n, m, max_pivots=caps[k])
        for f, a, b in zip(alone._fields, alone, res.lp(k)):
            if a is None:
                assert b is None, f
                continue
            assert a.shape == b.shape and a.dtype == b.dtype, (k, f, a.shape, b.shape)
            assert a.tobytes() == b.tobytes(), (k, f)
    perm = np.random.default_rng(3).permutation(len(lps))
    res2 = spx.batched.solve_ragged([lps[q] for q in perm], max_pivots=[caps[q] for q in perm])
    for j, q in enumerate(perm):
        for a, b in zip(res.lp(int(q)), res2.lp(j)):
            if a is not None:
                assert a.tobytes() == b.tobytes(), (j, q)


@pytest.mark.gpu
def test_launch_counts_reuse_and_empty(spx):
    for shapes in ([(8, 2)] * 3, [(8, 2), (20, 20)], [(100, 100), (128, 256), (3, 9000)],
                   [(4, 2), (99, 99), (400, 800), (256, 512)]):
        lps = [W.dense_lp(n, m, s) for s, (n, m) in enumerate(shapes)]
        spx.L.spx_launch_count(1)
        spx.batched.solve_ragged(lps, max_pivots=20)
        assert spx.L.spx_launch_count(1) == expected_launches(spx.L, shapes), shapes
    shapes = [(8, 2), (30, 30), (100, 100), (128, 256)]
    db = spx.batched.DeviceRaggedBatch(shapes, [50, 300, 2000, 2000])
    assert db.kernels == ["smem", "smem", "cluster", "cluster"] and db.launches == 4
    for seed in (1, 2):
        lps = [W.phase1_lp(n, m, seed * 10 + s) for s, (n, m) in enumerate(shapes)]
        db.upload(np.concatenate([flat_of(r, c) for r, c in lps]))
        db.run(spx.N.RULE_REFERENCE)
        res = db.result()
        for k, (rows, c) in enumerate(lps):
            o = oracle.solve_flat(flat_of(rows, c), rows.shape[0], c.shape[0], max_pivots=db.caps[k])
            assert (int(res.status[k]), int(res.npiv[k])) == (o.status, o.npiv)
            assert np.array_equal(bits(res.lp(k).tables[0]), bits(o.table)), (seed, k)
    empty = spx.batched.solve_ragged([], max_pivots=10)
    assert empty.status.shape == (0,) and empty.tables.shape == (0,) and empty.shapes.shape == (0, 3)
    with pytest.raises(ValueError, match="^LP 1: .*capacity"):
        spx.batched.solve_ragged([W.dense_lp(4, 2, 0), W.dense_lp(600, 800, 0)])


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded_worker(rank, world, port, out):
    import datetime
    import torch
    import torch.distributed as dist
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev, timeout=datetime.timedelta(seconds=120))
    try:
        from simplex_method_solver_b200.parallel import solve_ragged_sharded
        lps, caps = _mixed(90, 4, cap_max=500)
        start, count, res = solve_ragged_sharded(lps, max_pivots=caps, device=dev)
        out.put((rank, start, count, [[None if a is None else a.copy() for a in res.lp(k)] for k in range(count)]))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_over_gpus_concatenates_to_one_gpu(spx):
    import torch
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    lps, caps = _mixed(90, 4, cap_max=500)
    full = spx.batched.solve_ragged(lps, max_pivots=caps)
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_sharded_worker, args=(r, world, port, out), daemon=True) for r in range(world)]
    for p in procs:
        p.start()
    try:
        got = sorted(out.get(timeout=150) for _ in range(world))
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
    k = 0
    for rank, start, count, parts in got:
        assert start == k
        for j, one in enumerate(parts):
            for a, b in zip(one, full.lp(start + j)):
                if a is not None:
                    assert a.tobytes() == b.tobytes(), (rank, j)
        k += count
    assert k == len(lps)
