"""Batches of independent LPs of one shape, each solved whole inside one kernel.

Each LP is the reference's whole get_solution() loop
(/root/reference/src/simplex.py:179-199) with its tableau in shared memory:
  * "smem"    (K4, csrc/spx_batched.cu): one warp or one CTA per LP, up to
              ``spx_batched_max_cells()`` cells;
  * "cluster" (K7, csrc/spx_cluster.cu): one thread-block cluster of up to 16
              CTAs per LP, for mid-size LPs up to ``spx_cluster_size() > 0``.
``engine="auto"`` takes K4 for every shape K4 accepts and K7 above that.  Both
compute the same bits.  LPs never communicate, so a batch splits over GPUs by
contiguous ranges with no collective (see parallel.shard_range).
"""
from __future__ import annotations

from typing import NamedTuple, Optional

import numpy as np
import torch

from . import _native as N


class BatchResult(NamedTuple):
    status: np.ndarray            # [B] int32: N.OPTIMAL / N.INCORRECT / N.NOCONV / N.CAP
    npiv: np.ndarray              # [B] int32
    x: np.ndarray                 # [B, m]
    obj: np.ndarray               # [B]  function[0]*x1 + function[1]*x2  (simplex.py:49)
    tables: np.ndarray            # [B, cells] final reference-flat tables
    rowlab: np.ndarray            # [B, m] int32 label codes
    collab: np.ndarray            # [B, n] int32
    trace: Optional[np.ndarray]   # [B, max_pivots, 2] int32
    snaps: Optional[np.ndarray]   # [B, max_pivots+1, cells]


ENGINES = ("auto", "smem", "cluster")
_INT32_MAX = (1 << 31) - 1


def _cluster_capacity_text(n: int, m: int) -> str:
    L = N.load()
    if L.spx_cluster_size(1, m) == 0:
        return f"at most {max(k for k in range(1, m + 1) if L.spx_cluster_size(1, k))} columns fit one cluster"
    lo, hi = 1, 1 << 20                        # largest n with spx_cluster_size(n, m) > 0
    while lo < hi:
        mid = (lo + hi + 1) // 2
        lo, hi = (mid, hi) if L.spx_cluster_size(mid, m) else (lo, mid - 1)
    return f"at m = {m} one cluster of 16 CTAs holds at most n = {lo} rows"


def kernel_for(n: int, m: int, engine: str = "auto") -> str:
    """"smem" (K4) or "cluster" (K7) for an n x m LP; ValueError when the engine cannot take it."""
    if engine not in ENGINES:
        raise ValueError(f"unknown engine {engine!r}; one of {ENGINES}")
    if not (1 <= n <= _INT32_MAX and 1 <= m <= _INT32_MAX):
        raise ValueError(f"bad shape {n} x {m}")
    L = N.load()
    cells = n * (m + 1) + m
    if engine == "smem" or (engine == "auto" and cells <= L.spx_batched_max_cells()):
        if cells > L.spx_batched_max_cells():
            raise ValueError(f"{cells} cells per LP exceed the shared-memory limit of one CTA "
                             f"({L.spx_batched_max_cells()}); use engine='cluster' or 'auto'")
        return "smem"
    if L.spx_cluster_size(n, m) == 0:
        raise ValueError(f"a {n} x {m} LP ({cells} cells) exceeds the capacity of the cluster solver: "
                         f"{_cluster_capacity_text(n, m)}; use SimplexMethod / DeviceTableau for large tableaus")
    return "cluster"


class DeviceBatch:
    """Device buffers for one batch shape; reusable across solves (bench / serving).

    ``kernel`` is "smem" (K4) or "cluster" (K7), chosen by ``kernel_for(n, m, engine)``.
    """

    def __init__(self, B: int, n: int, m: int, max_pivots: int = 64, trace: bool = True,
                 snapshots: bool = False, device=None, engine: str = "auto"):
        N.lib()
        self.device = torch.device(device if device is not None else "cuda")
        self.B, self.n, self.m, self.max_pivots = int(B), int(n), int(m), int(max_pivots)
        self.cells = n * (m + 1) + m
        self.kernel = kernel_for(self.n, self.m, engine)
        dev = self.device
        Bq = max(self.B, 1)
        self.T = torch.empty((Bq, self.cells), dtype=torch.float64, device=dev)
        self.x = torch.empty((Bq, m), dtype=torch.float64, device=dev)
        self.obj = torch.empty(Bq, dtype=torch.float64, device=dev)
        self.status = torch.empty(Bq, dtype=torch.int32, device=dev)
        self.npiv = torch.empty(Bq, dtype=torch.int32, device=dev)
        self.rowlab = torch.empty((Bq, m), dtype=torch.int32, device=dev)
        self.collab = torch.empty((Bq, n), dtype=torch.int32, device=dev)
        self.trace = (torch.zeros((Bq, max(self.max_pivots, 1), 2), dtype=torch.int32, device=dev)
                      if trace else None)
        self.snaps = (torch.empty((Bq, self.max_pivots + 1, self.cells), dtype=torch.float64, device=dev)
                      if snapshots else None)

    def upload(self, tables, non_blocking: bool = False):
        """tables: [B, cells] fp64 numpy array or (pinned) CPU tensor."""
        src = torch.from_numpy(tables) if isinstance(tables, np.ndarray) else tables
        self.T[: self.B].copy_(src, non_blocking=non_blocking)

    def run(self, rule: int = N.RULE_REFERENCE):
        """Launch the solver on the resident batch (asynchronous on the current stream)."""
        with torch.cuda.device(self.device):
            entry = "spx_solve_batched" if self.kernel == "smem" else "spx_solve_batched_cluster"
            N.call(entry, self.T.data_ptr(), self.B, self.n, self.m, rule, self.max_pivots, self.x.data_ptr(), self.obj.data_ptr(), self.status.data_ptr(),
                   self.npiv.data_ptr(), self.rowlab.data_ptr(), self.collab.data_ptr(),
                   N.ptr(self.trace), N.ptr(self.snaps),
                   torch.cuda.current_stream(self.device).cuda_stream)

    def result(self) -> BatchResult:
        B = self.B
        g = lambda t: None if t is None else t[:B].cpu().numpy()  # noqa: E731
        return BatchResult(g(self.status), g(self.npiv), g(self.x), g(self.obj), g(self.T),
                           g(self.rowlab), g(self.collab), g(self.trace), g(self.snaps))


def solve_batched(tables, n: int, m: int, max_pivots: int = 64, rule: str = "reference",
                  trace: bool = True, snapshots: bool = False, device=None, engine: str = "auto") -> BatchResult:
    """Solve B independent LPs of one shape.

    tables: [B, cells] reference-flat fp64 (rows ``[a_1..a_m, b]`` x n, then the m
    function coefficients) — the flattened arguments of
    ``SimplexMethod(constraints, function)`` for each LP.
    engine: "auto" (K4 when the LP fits one CTA, else K7), "smem" (K4) or "cluster" (K7).
    """
    tables = np.ascontiguousarray(np.asarray(tables, dtype=np.float64))
    if tables.ndim != 2 or tables.shape[1] != n * (m + 1) + m:
        raise ValueError("tables must be [B, n*(m+1)+m]")
    db = DeviceBatch(tables.shape[0], n, m, max_pivots, trace, snapshots, device, engine)
    if db.B == 0:
        z = np.zeros
        return BatchResult(z(0, np.int32), z(0, np.int32), z((0, m)), z(0), z((0, db.cells)),
                           z((0, m), np.int32), z((0, n), np.int32),
                           z((0, max_pivots, 2), np.int32) if trace else None,
                           z((0, max_pivots + 1, db.cells)) if snapshots else None)
    db.upload(tables)
    db.run(N.RULES[rule])
    return db.result()
