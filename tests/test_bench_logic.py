"""CPU (gloo, world 2) tests of bench.py's multi-GPU bookkeeping — the parts that deadlocked or crashed on real GPUs
before they were covered here: the "late"-LP preflight (trace + b + f + body checksum against the oracle golden, with the
same collectives on every rank whatever happens on one of them) and the int64 transport of unsigned checksums; on a GPU,
the arrays --dump-outputs writes."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_checksum_transport_is_bit_preserving():
    import bench
    for v in (0, 5, (1 << 63) - 1, 1 << 63, (1 << 64) - 1, 0xDEADBEEFCAFEF00D):
        t = torch.tensor([bench.as_i64(v)], dtype=torch.int64)
        assert int(t.item()) & 0xFFFFFFFFFFFFFFFF == v
    a, b = 0xF000000000000001, 0x2000000000000005                   # the sum wraps mod 2^64 in int64 too
    s = torch.tensor([bench.as_i64(a)], dtype=torch.int64) + torch.tensor([bench.as_i64(b)], dtype=torch.int64)
    assert int(s.item()) & 0xFFFFFFFFFFFFFFFF == (a + b) % (1 << 64)


def _preflight_worker(rank, world, port, fail_rank, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import datetime
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=120))
    try:
        import bench
        from cpu_shard_ops import CpuShardOps
        from simplex_method_solver_b200 import parallel as P

        class CpuFused(P.ShardedTableau):
            """FusedShardedTableau's surface on the numpy stand-in kernels (same shards, same replicated pieces)."""

            def __init__(self, n, m, rank, world, device, trace_capacity=0, depth=8):
                super().__init__(n, m, rank, world, device="cpu", trace_capacity=trace_capacity, ops=CpuShardOps(),
                                 lookahead=False)

            def local_body(self):
                # what happened on hardware: ONE rank's digest raised (an unsigned checksum >= 2^63 into an int64
                # tensor) after the ranks had pivoted together
                if self.rank == fail_rank:
                    raise RuntimeError("injected failure on one rank")
                return super().local_body()

            def close(self):
                pass

        ok, changes, why = bench.late_lp_preflight(CpuFused, rank, world, torch.device("cpu"), dist)
        out.put((rank, ok, changes, why))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("fail_rank", [-1, 1])
def test_late_lp_preflight_under_gloo(fail_rank):
    """All ranks agree on the verdict, with and without a failure injected on ONE rank (which used to leave the other
    ranks waiting in a collective the failed rank never entered)."""
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_preflight_worker, args=(r, world, port, fail_rank, out), daemon=True) for r in range(world)]
    for p in procs:
        p.start()
    try:
        got = sorted(out.get(timeout=240) for _ in range(world))
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
    if fail_rank < 0:
        assert [g[1] for g in got] == [True, True], got
        assert got[0][2] == got[1][2] == 186                          # owner changes of the entering column on 2 ranks
    else:
        assert [g[1] for g in got] == [False, False]
        assert "injected failure" in got[fail_rank][3]


@pytest.mark.gpu
def test_dump_outputs_equal_the_oracle(tmp_path):
    """bench.py --dump-outputs on a small tableau: every array it writes is float64 and equals, bit for bit, what the
    oracle holds after the same pivots."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import bench
    import oracle
    from simplex_method_solver_b200 import workloads as W
    from simplex_method_solver_b200.engine import DeviceTableau
    n, m, k, step = 96, 700, 40, 16
    rows, c = W.dense_lp(n, m, seed=3)
    tab = DeviceTableau(n, m, device="cuda:0", trace_capacity=k + 64)
    tab.load(rows, c, max_pivots=k + 64)
    st, npiv = tab.solve(chunk=step, stop_after=k)
    assert npiv == k
    bench.dump_outputs(str(tmp_path / "out"), tab, st, npiv, step)
    got = {p.stem: np.load(p) for p in (tmp_path / "out").glob("*.npy")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(a.nbytes for a in got.values()) < 64 << 20
    o = oracle.solve(rows, c, max_pivots=k)
    body = o.table[: n * (m + 1)].reshape(n, m + 1)
    assert got["status"].tolist() == [st, k]
    assert got["trace"].tolist() == o.trace[k - step:].tolist()
    assert got["b"].tobytes() == body[:, m].tobytes() and got["f_row"].tobytes() == o.table[n * (m + 1):].tobytes()
    idx = got["body_sample_index"].astype(np.int64)
    assert (np.diff(idx) > 0).all() and idx[-1] < n * m
    assert got["body_sample"].tobytes() == body[:, :m].reshape(-1)[idx].tobytes()
    assert got["x"].tobytes() == o.x.tobytes() and got["objective"].tobytes() == np.array([o.obj2, o.objm]).tobytes()
    assert got["row_labels"].tolist() == o.rowlab.tolist() and got["column_labels"].tolist() == o.collab.tolist()


def test_price_engine_choice():
    """Which pricing engine the column-sharded fused loop uses (parallel.choose_price_engine): by world size unless forced."""
    from simplex_method_solver_b200.parallel import choose_price_engine as ch
    assert [ch(True, w) for w in (1, 2, 8, 16)] == [1, 1, 1, 1]                       # the shipped default: never
    assert [ch(True, w, "", 8) for w in (1, 2, 4, 7, 8, 16)] == [1, 1, 1, 1, 2, 2]
    assert ch(False, 8) == 0 and ch(False, 8, "persistent") == 0
    assert ch("per-pass", 8) == 1 and ch("persistent", 1) == 2
    assert ch(True, 2, "persistent") == 2 and ch(True, 8, "per-pass", 8) == 1 and ch(True, 8, "nonsense", 8) == 2
    assert ch("persistent", 8, "per-pass") == 2           # an explicit argument beats the environment
