"""Batches of independent LPs, each solved whole inside one kernel: of one shape (``solve_batched``,
``DeviceBatch``) or of any mix of shapes (``solve_ragged``, ``DeviceRaggedBatch``).

Each LP is the reference's whole get_solution() loop
(/root/reference/src/simplex.py:179-199) with its tableau in shared memory:
  * "smem"    (K4, csrc/spx_batched.cu): one warp or one CTA per LP, up to
              ``spx_batched_max_cells()`` cells;
  * "cluster" (K7, csrc/spx_cluster.cu): one thread-block cluster of up to 16
              CTAs per LP, for mid-size LPs up to ``spx_cluster_size() > 0``;
  * "global"  (K8, csrc/spx_global.cu): one cluster per LP with the table left in
              global memory, for LPs up to ``spx_global_min_cluster_size() > 0``
              (only when asked for: ``engine="auto"`` never routes to it).
``engine="auto"`` takes K4 for every shape K4 accepts and K7 above that;
``engine="auto_global"`` does the same and takes K8 above K7's capacity.  All three
compute the same bits.  LPs never communicate, so a batch splits over GPUs by
contiguous ranges with no collective (see parallel.shard_range).

A ragged batch is packed in batch order (LP k's table, x, labels, trace and snapshots
start at prefix sums over LPs 0..k-1, see include/spx_b200.h) and solved by one plan of
at most twelve launches: K4 warp mode, K4 CTA mode, one K7 launch per cluster size, one
K8 launch per smallest cluster size that holds its LPs.

Warm start: a batch's final tables are dictionaries, so they can be continued (``resume``, e.g. after
``SPX_CAP``) or re-optimised after new right-hand sides and costs (``change`` then ``resume``; ``resolve``
does both from a host result).  The change is exact to the bit (include/spx_b200.h, spx_warm_change_*).
"""
from __future__ import annotations

from typing import NamedTuple, Optional, Sequence, Union

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


class Sensitivity(NamedTuple):
    """Sensitivity report of optimal LPs (spx_sensitivity_*, include/spx_b200.h): the LP is "minimise c.x subject to
    b + A x >= 0 and x >= 0", constraint k's slack is y_k.  Every output of an LP that is not optimal is NaN.
    Ranges are (allowable decrease, allowable increase), +inf when unbounded."""
    dual: np.ndarray              # [B, n] shadow price of each constraint, d f* / d b_k
    slack: np.ndarray             # [B, n] value of each constraint's slack y_k at the optimum
    reduced_cost: np.ndarray      # [B, m]
    rhs_range: np.ndarray         # [B, n, 2] how far b_k may move before the optimal basis changes
    cost_range: np.ndarray        # [B, m, 2] how far c_k may move before the optimal basis changes
    optimal: np.ndarray           # [B] bool


class _SensOut:
    """Device outputs of one sensitivity call: nc per-constraint and nv per-variable entries."""

    def __init__(self, nc: int, nv: int, device):
        f64, q = torch.float64, (lambda k: max(k, 1))  # noqa: E731
        self.nc, self.nv = nc, nv
        self.t = [torch.empty(q(nc), dtype=f64, device=device), torch.empty(q(nc), dtype=f64, device=device),
                  torch.empty(q(nv), dtype=f64, device=device), torch.empty(q(2 * nc), dtype=f64, device=device),
                  torch.empty(q(2 * nv), dtype=f64, device=device)]

    def ptrs(self):
        return [t.data_ptr() for t in self.t]

    def host(self):
        nc, nv = self.nc, self.nv
        return [t[:k].cpu().numpy() for t, k in zip(self.t, (nc, nc, nv, 2 * nc, 2 * nv))]


def _sens_uniform(T, status, rowlab, collab, B: int, n: int, m: int, device) -> Sensitivity:
    out = _SensOut(B * n, B * m, device)
    with torch.cuda.device(device):
        N.call("spx_sensitivity_batched", T.data_ptr(), B, n, m, status.data_ptr(), rowlab.data_ptr(),
               collab.data_ptr(), *out.ptrs(), torch.cuda.current_stream(device).cuda_stream)
    dual, slack, rc, rr, cr = out.host()
    return Sensitivity(dual.reshape(B, n), slack.reshape(B, n), rc.reshape(B, m), rr.reshape(B, n, 2),
                       cr.reshape(B, m, 2), status[:B].cpu().numpy() == N.OPTIMAL)


ENGINES = ("auto", "smem", "cluster", "global", "auto_global")
ENGINE_CODES = {"auto": N.ENGINE_AUTO, "smem": N.ENGINE_SMEM, "cluster": N.ENGINE_CLUSTER, "global": N.ENGINE_GLOBAL,
                "auto_global": N.ENGINE_AUTO_GLOBAL}
_INT32_MAX = (1 << 31) - 1


def kernel_for(n: int, m: int, engine: str = "auto") -> str:
    """"smem" (K4), "cluster" (K7) or "global" (K8) for an n x m LP; ValueError when the engine cannot take it.

    The library's routing rule, ``spx_batched_route`` (include/spx_b200.h): "auto" is K4 when
    ``spx_batched_fits(n, m)`` (at most ``spx_batched_max_cells()`` cells, and one CTA's shared memory holds the LP),
    else K7.  "auto_global" is "auto" with K8 above K7's capacity: K4 when it fits, else K7 when
    ``spx_cluster_size(n, m) > 0``, else K8 (the routing of ragged batches that mix every size).
    """
    if engine not in ENGINES:
        raise ValueError(f"unknown engine {engine!r}; one of {ENGINES}")
    if not (1 <= n <= _INT32_MAX and 1 <= m <= _INT32_MAX):
        raise ValueError(f"bad shape {n} x {m}")
    L = N.load()
    code = L.spx_batched_route(n, m, ENGINE_CODES[engine])
    if code < 0:
        raise ValueError(L.spx_last_error().decode(errors="replace"))
    return {N.ENGINE_SMEM: "smem", N.ENGINE_CLUSTER: "cluster", N.ENGINE_GLOBAL: "global"}[code]


_ENTRIES = {"smem": "spx_solve_batched", "cluster": "spx_solve_batched_cluster", "global": "spx_solve_batched_global"}


_ENGINE_OF_KERNEL = {"smem": N.ENGINE_SMEM, "cluster": N.ENGINE_CLUSTER, "global": N.ENGINE_GLOBAL}


def _per_lp(a, B: int, k: int, name: str) -> np.ndarray:
    """[B, k] or [k] (broadcast over the batch) -> contiguous fp64 [B, k]."""
    a = np.asarray(a, dtype=np.float64)
    if a.shape == (k,):
        a = np.broadcast_to(a, (B, k))
    if a.shape != (B, k):
        raise ValueError(f"{name} must be [{B}, {k}] or [{k}], got shape {a.shape}")
    return np.ascontiguousarray(a)


def _check_finite(a: Optional[np.ndarray], what: str, starts: Optional[np.ndarray] = None) -> None:
    """A non-finite entry of `a` is a ValueError naming its LP: a is [B, k], one row per LP, or with `starts` packed,
    LP k's entries from starts[k] on (n, m >= 1: no LP's slice is empty).  None passes."""
    bad = np.flatnonzero(~np.isfinite(a)) if a is not None else []
    if len(bad):
        lp = bad[0] // a.shape[1] if starts is None else np.searchsorted(starts, bad[0], side="right") - 1
        raise ValueError(f"LP {int(lp)}: {what} is not finite")


def _check_labels(rowlab: np.ndarray, collab: np.ndarray) -> None:
    """rowlab [B, m], collab [B, n]: each LP's labels must be a permutation of 0..n+m-1."""
    n, m = collab.shape[1], rowlab.shape[1]
    lab = np.sort(np.concatenate([rowlab, collab], axis=1), axis=1)
    bad = np.flatnonzero((lab != np.arange(n + m)).any(axis=1))
    if bad.size:
        raise ValueError(f"LP {int(bad[0])}: labels are not a permutation of 0..{n + m - 1}")


def _check_ragged_labels(rowlab: np.ndarray, collab: np.ndarray, shapes: np.ndarray, xm, xn) -> None:
    """packed labels: LP k's rowlab at xm[k], collab at xn[k] must be a permutation of 0..n_k+m_k-1"""
    for k, (n, m) in enumerate(np.asarray(shapes, dtype=np.int64).reshape(-1, 2)):
        n, m, a, b = int(n), int(m), int(xm[k]), int(xn[k])
        lab = np.sort(np.concatenate([rowlab[a: a + m], collab[b: b + n]]))
        if not np.array_equal(lab, np.arange(n + m)):
            raise ValueError(f"LP {k}: labels are not a permutation of 0..{n + m - 1}")


def _empty_batch(n: int, m: int, max_pivots: int, trace: bool, snapshots: bool) -> BatchResult:
    z, cells = np.zeros, n * (m + 1) + m
    return BatchResult(z(0, np.int32), z(0, np.int32), z((0, m)), z(0), z((0, cells)), z((0, m), np.int32),
                       z((0, n), np.int32), z((0, max_pivots, 2), np.int32) if trace else None,
                       z((0, max_pivots + 1, cells)) if snapshots else None)


class DeviceBatch:
    """Device buffers for one batch shape; reusable across solves (bench / serving).

    ``kernel`` is "smem" (K4), "cluster" (K7) or "global" (K8), chosen by ``kernel_for(n, m, engine)``.
    ``cluster_size`` is the CTAs per LP a K8 ``run`` launches on this device (None for K4 and K7).
    """

    def __init__(self, B: int, n: int, m: int, max_pivots: int = 64, trace: bool = True,
                 snapshots: bool = False, device=None, engine: str = "auto"):
        N.lib()
        self.device = torch.device(device if device is not None else "cuda")
        self.B, self.n, self.m, self.max_pivots = int(B), int(n), int(m), int(max_pivots)
        self.cells = n * (m + 1) + m
        self.kernel = kernel_for(self.n, self.m, engine)
        dev = self.device
        self.cluster_size = None
        if self.kernel == "global":
            with torch.cuda.device(dev):
                self.cluster_size = int(N.lib().spx_global_cluster_size(self.n, self.m, self.B))
            if self.cluster_size <= 0:
                raise N.SpxError(f"spx_global_cluster_size failed: {N.lib().spx_last_error().decode(errors='replace')}")
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
            entry = _ENTRIES[self.kernel]
            N.call(entry, self.T.data_ptr(), self.B, self.n, self.m, rule, self.max_pivots, self.x.data_ptr(), self.obj.data_ptr(), self.status.data_ptr(),
                   self.npiv.data_ptr(), self.rowlab.data_ptr(), self.collab.data_ptr(),
                   N.ptr(self.trace), N.ptr(self.snaps),
                   torch.cuda.current_stream(self.device).cuda_stream)

    def upload_labels(self, rowlab, collab, non_blocking: bool = False):
        """Set the labels a ``change`` and a ``resume`` start from: rowlab [B, m] and collab [B, n] int label codes
        of final tables (e.g. a host ``BatchResult``'s).  Labels that are not a permutation of 0..n+m-1 are a
        ValueError naming the LP."""
        rowlab = np.ascontiguousarray(rowlab, dtype=np.int32)
        collab = np.ascontiguousarray(collab, dtype=np.int32)
        if rowlab.shape != (self.B, self.m) or collab.shape != (self.B, self.n):
            raise ValueError(f"rowlab must be [{self.B}, {self.m}] and collab [{self.B}, {self.n}], got "
                             f"{rowlab.shape} and {collab.shape}")
        _check_labels(rowlab, collab)
        self.rowlab[: self.B].copy_(torch.from_numpy(rowlab), non_blocking=non_blocking)
        self.collab[: self.B].copy_(torch.from_numpy(collab), non_blocking=non_blocking)

    def change(self, rhs_delta=None, cost_delta=None):
        """Apply new right-hand sides b + rhs_delta and costs c + cost_delta to the resident final tables, in
        place, with the labels the last ``run``, ``resume`` or ``upload_labels`` left (``spx_warm_change_batched``, exact to the bit).
        rhs_delta: [B, n] or [n] (broadcast over the batch); cost_delta: [B, m] or [m]; either may be None.
        A non-finite delta is a ValueError naming the LP.  Asynchronous on the current stream."""
        B, n, m = self.B, self.n, self.m
        db = None if rhs_delta is None else _per_lp(rhs_delta, B, n, "rhs_delta")
        dc = None if cost_delta is None else _per_lp(cost_delta, B, m, "cost_delta")
        _check_finite(db, "rhs_delta")
        _check_finite(dc, "cost_delta")
        if B == 0 or (db is None and dc is None):
            return
        up = lambda a: None if a is None else torch.from_numpy(a).to(self.device)  # noqa: E731
        d_db, d_dc = up(db), up(dc)
        with torch.cuda.device(self.device):
            N.call("spx_warm_change_batched", self.T.data_ptr(), B, n, m, self.rowlab.data_ptr(),
                   self.collab.data_ptr(), N.ptr(d_db), N.ptr(d_dc), torch.cuda.current_stream(self.device).cuda_stream)

    def resume(self, function, rule: int = N.RULE_REFERENCE):
        """Continue every LP from its resident table and labels for up to ``max_pivots`` more pivots, on this
        batch's engine (``spx_warm_solve_batched``).  function: [B, m] or [m], the LPs' current costs, used only
        for ``obj``.  Trace and snapshots count from 0 again.  Asynchronous on the current stream."""
        fn = _per_lp(function, self.B, self.m, "function")
        self._function = torch.from_numpy(fn).to(self.device) if self.B else None    # alive until the kernel ran
        with torch.cuda.device(self.device):
            N.call("spx_warm_solve_batched", _ENGINE_OF_KERNEL[self.kernel], self.T.data_ptr(), self.B, self.n,
                   self.m, rule, self.max_pivots, N.ptr(self._function), self.x.data_ptr(), self.obj.data_ptr(),
                   self.status.data_ptr(), self.npiv.data_ptr(), self.rowlab.data_ptr(), self.collab.data_ptr(),
                   N.ptr(self.trace), N.ptr(self.snaps), torch.cuda.current_stream(self.device).cuda_stream)

    def sensitivity(self) -> Sensitivity:
        """Sensitivity report of the final tables the last ``run`` left (K4, K7 and K8 alike); synchronises."""
        return _sens_uniform(self.T, self.status, self.rowlab, self.collab, self.B, self.n, self.m, self.device)

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
    engine: "auto" (K4 when the LP fits one CTA, else K7), "smem" (K4), "cluster" (K7) or "global" (K8).
    """
    tables = np.ascontiguousarray(np.asarray(tables, dtype=np.float64))
    if tables.ndim != 2 or tables.shape[1] != n * (m + 1) + m:
        raise ValueError("tables must be [B, n*(m+1)+m]")
    db = DeviceBatch(tables.shape[0], n, m, max_pivots, trace, snapshots, device, engine)
    if db.B == 0:
        return _empty_batch(n, m, max_pivots, trace, snapshots)
    db.upload(tables)
    db.run(N.RULES[rule])
    return db.result()


# ---------------------------------------------------------------------------- ragged batches
# the plan spx_ragged_plan writes (csrc/spx_common.cuh: RaggedPlan, RaggedLaunch, RaggedLp)
_LAUNCH = np.dtype([("kernel", "<i4"), ("S", "<i4"), ("threads", "<i4"), ("per_cta", "<i4"), ("smem", "<i8"),
                    ("first", "<i8"), ("count", "<i8"), ("slot_doubles", "<i8"), ("pick_S", "<i4"), ("reserved", "<i4")])
_HEADER = np.dtype([("magic", "<u4"), ("abi", "<i4"), ("B", "<i8"), ("engine", "<i4"), ("nlaunch", "<i4"),
                    ("totals", "<i8", 5), ("lp_offset", "<i8"), ("order_offset", "<i8"), ("launch", _LAUNCH, 12)])
_LP = np.dtype([("n", "<i4"), ("m", "<i4"), ("max_pivots", "<i4"), ("cells", "<i4"), ("t", "<i8"), ("xm", "<i8"),
                ("xn", "<i8"), ("tr", "<i8"), ("sn", "<i8")])
LAUNCH_KINDS = ("warp", "cta", "cluster", "global")


class RaggedPlan(NamedTuple):
    plan: np.ndarray              # the plan bytes (uint8), as spx_ragged_plan wrote them
    totals: np.ndarray            # [5] packed lengths: T, x (= rowlab), collab, trace pairs, snap
    lps: np.ndarray               # [B] descriptors: n, m, max_pivots, cells and the offsets t, xm, xn, tr, sn
    offsets: np.ndarray           # [B, 5] int64: the offsets t, xm, xn, tr, sn of each LP (RaggedResult.offsets)
    launches: list                # per launch: dict(kind, S, threads, smem, lps = LP indices in launch order);
    #                               for kind "global" S is the planned S (S_min, or SPX_OPT_CLUSTER_SIZE)


def ragged_plan(shapes, max_pivots, engine: str = "auto") -> RaggedPlan:
    """Host only: the library's plan for LPs of `shapes` [B, 2] (n, m) with caps `max_pivots` [B]."""
    if engine not in ENGINE_CODES:
        raise ValueError(f"unknown engine {engine!r}; one of {tuple(ENGINE_CODES)}")
    L = N.load()
    shapes = np.asarray(shapes, dtype=np.int64).reshape(-1, 2)
    B = shapes.shape[0]
    caps = np.broadcast_to(np.asarray(max_pivots, dtype=np.int64), (B,))
    if not (np.all(np.abs(shapes) <= _INT32_MAX) and np.all(np.abs(caps) <= _INT32_MAX)):
        raise ValueError("shapes and caps must fit int32")
    h = np.ascontiguousarray(np.concatenate([shapes, caps[:, None]], axis=1), dtype=np.int32)
    nbytes = int(L.spx_ragged_plan_bytes(B))
    plan = np.zeros(max(nbytes, 16), dtype=np.uint8)
    totals = np.zeros(5, dtype=np.int64)
    rc = L.spx_ragged_plan(h.ctypes.data, B, ENGINE_CODES[engine], plan.ctypes.data, nbytes, totals.ctypes.data)
    if rc != 0:
        raise ValueError(L.spx_last_error().decode(errors="replace"))
    hd = plan[: _HEADER.itemsize].view(_HEADER)[0]
    lo, oo = int(hd["lp_offset"]), int(hd["order_offset"])
    lps = plan[lo: lo + B * _LP.itemsize].view(_LP)
    order = plan[oo: oo + 4 * B].view("<i4")
    launches = []
    for q in range(int(hd["nlaunch"])):
        la = hd["launch"][q]
        f, c = int(la["first"]), int(la["count"])
        launches.append({"kind": LAUNCH_KINDS[int(la["kernel"])], "S": int(la["S"]), "threads": int(la["threads"]),
                         "smem": int(la["smem"]), "lps": order[f: f + c].copy()})
    offsets = np.stack([lps["t"], lps["xm"], lps["xn"], lps["tr"], lps["sn"]], axis=1).astype(np.int64)
    return RaggedPlan(plan, totals, lps, offsets, launches)


class RaggedResult(NamedTuple):
    """Results of a ragged batch, packed in batch order at the plan's offsets."""
    status: np.ndarray            # [B] int32
    npiv: np.ndarray              # [B] int32
    x: np.ndarray                 # [sum m]
    obj: np.ndarray               # [B]
    tables: np.ndarray            # [sum cells] final reference-flat tables
    rowlab: np.ndarray            # [sum m] int32
    collab: np.ndarray            # [sum n] int32
    trace: Optional[np.ndarray]   # [sum max_pivots, 2] int32
    snaps: Optional[np.ndarray]   # [sum (max_pivots+1)*cells]
    shapes: np.ndarray            # [B, 3] int64: n, m, max_pivots
    offsets: np.ndarray           # [B, 5] int64: first cell / x / collab / trace pair / snapshot cell of each LP

    def lp(self, k: int) -> BatchResult:
        """LP k alone, with the shapes and dtypes ``solve_batched(flat_k[None], n_k, m_k, max_pivots=cap_k)`` returns."""
        n, m, cap = (int(v) for v in self.shapes[k])
        t, xm, xn, tr, sn = (int(v) for v in self.offsets[k])
        cells = n * (m + 1) + m
        trace = None
        if self.trace is not None:        # DeviceBatch keeps at least one (zeroed) pair per LP
            trace = self.trace[tr: tr + cap][None] if cap > 0 else np.zeros((1, 1, 2), dtype=np.int32)
        return BatchResult(self.status[k: k + 1], self.npiv[k: k + 1], self.x[xm: xm + m][None], self.obj[k: k + 1],
                           self.tables[t: t + cells][None], self.rowlab[xm: xm + m][None],
                           self.collab[xn: xn + n][None], trace,
                           None if self.snaps is None else self.snaps[sn: sn + (cap + 1) * cells].reshape(1, cap + 1, cells))


class RaggedSensitivity(NamedTuple):
    """Sensitivity report of a ragged batch, packed in batch order: per-constraint outputs at the prefix sums of n
    (as ``collab``), per-variable outputs at the prefix sums of m (as ``x``)."""
    dual: np.ndarray              # [sum n]
    slack: np.ndarray             # [sum n]
    reduced_cost: np.ndarray      # [sum m]
    rhs_range: np.ndarray         # [sum n, 2]
    cost_range: np.ndarray        # [sum m, 2]
    optimal: np.ndarray           # [B] bool
    shapes: np.ndarray            # [B, 3] int64: n, m, max_pivots
    offsets: np.ndarray           # [B, 5] int64, as RaggedResult.offsets

    def lp(self, k: int) -> Sensitivity:
        """LP k alone, with the shapes ``DeviceBatch.sensitivity()`` gives for a batch of that one LP."""
        n, m = int(self.shapes[k, 0]), int(self.shapes[k, 1])
        xm, xn = int(self.offsets[k, 1]), int(self.offsets[k, 2])
        return Sensitivity(self.dual[xn: xn + n][None], self.slack[xn: xn + n][None],
                           self.reduced_cost[xm: xm + m][None], self.rhs_range[xn: xn + n][None],
                           self.cost_range[xm: xm + m][None], self.optimal[k: k + 1])


def _sens_ragged(T, h_plan: np.ndarray, d_plan, status, rowlab, collab, B: int, totals, shapes, offsets,
                 device) -> RaggedSensitivity:
    out = _SensOut(int(totals[2]), int(totals[1]), device)
    with torch.cuda.device(device):
        N.call("spx_sensitivity_ragged", T.data_ptr(), h_plan.ctypes.data, d_plan.data_ptr(), status.data_ptr(),
               rowlab.data_ptr(), collab.data_ptr(), *out.ptrs(), torch.cuda.current_stream(device).cuda_stream)
    dual, slack, rc, rr, cr = out.host()
    return RaggedSensitivity(dual, slack, rc, rr.reshape(-1, 2), cr.reshape(-1, 2),
                             status[:B].cpu().numpy() == N.OPTIMAL, shapes.copy(), offsets.copy())


def _caps(max_pivots: Union[int, Sequence[int]], B: int) -> np.ndarray:
    caps = np.asarray(max_pivots, dtype=np.int64)
    if caps.ndim == 0:
        caps = np.full(B, int(caps), dtype=np.int64)
    if caps.shape != (B,):
        raise ValueError(f"max_pivots must be an int or one int per LP ({B}), got shape {caps.shape}")
    bad = np.flatnonzero(caps < 0)
    if bad.size:
        raise ValueError(f"LP {int(bad[0])}: max_pivots = {int(caps[bad[0]])} must be >= 0")
    return caps


def kernels_for(shapes, engine: str = "auto") -> list:
    """``kernel_for`` of every LP; its ValueError is prefixed with the index of the first LP it rejects."""
    shapes = np.asarray(shapes, dtype=np.int64).reshape(-1, 2)
    if shapes.shape[0] == 0:
        return []
    uniq, first, inv = np.unique(shapes, axis=0, return_index=True, return_inverse=True)
    kinds = [None] * len(uniq)
    for u in np.argsort(first, kind="stable"):     # in batch order, so the first bad LP is named
        n, m = (int(v) for v in uniq[u])
        try:
            kinds[u] = kernel_for(n, m, engine)
        except ValueError as e:
            raise ValueError(f"LP {int(first[u])}: {e}") from None
    return [kinds[i] for i in inv.reshape(-1)]


class DeviceRaggedBatch:
    """Device buffers and the plan of one ragged batch; reusable across solves (as ``DeviceBatch``).

    shapes: [B] (n, m) pairs; max_pivots: an int or one int per LP.  ``kernels`` is each LP's
    "smem" (K4), "cluster" (K7) or "global" (K8), ``launches`` the number of kernel launches of one
    ``run`` and ``cluster_sizes`` the CTAs per LP of each launch on this device (1 for K4).
    """

    def __init__(self, shapes, max_pivots: Union[int, Sequence[int]] = 64, trace: bool = True,
                 snapshots: bool = False, device=None, engine: str = "auto"):
        N.lib()
        self.device = torch.device(device if device is not None else "cuda")
        self.shapes2 = np.asarray(shapes, dtype=np.int64).reshape(-1, 2)
        self.B = int(self.shapes2.shape[0])
        self.caps = _caps(max_pivots, self.B)
        self.kernels = kernels_for(self.shapes2, engine)
        self.plan = ragged_plan(self.shapes2, self.caps, engine)
        self.launches = len(self.plan.launches)
        L = N.lib()
        with torch.cuda.device(self.device):
            self.cluster_sizes = [int(L.spx_ragged_cluster_size(self.plan.plan.ctypes.data, q))
                                  for q in range(self.launches)]
        if any(S <= 0 for S in self.cluster_sizes):
            raise N.SpxError(f"spx_ragged_cluster_size failed: {L.spx_last_error().decode(errors='replace')}")
        self.shapes = np.concatenate([self.shapes2, self.caps[:, None]], axis=1)
        self.offsets = self.plan.offsets
        tot = [int(v) for v in self.plan.totals]
        dev, f64, i32 = self.device, torch.float64, torch.int32
        q = lambda k: max(k, 1)  # noqa: E731
        self.d_plan = torch.from_numpy(self.plan.plan).to(dev)      # uploaded once
        self.T = torch.empty(q(tot[0]), dtype=f64, device=dev)
        self.x = torch.empty(q(tot[1]), dtype=f64, device=dev)
        self.obj = torch.empty(q(self.B), dtype=f64, device=dev)
        self.status = torch.empty(q(self.B), dtype=i32, device=dev)
        self.npiv = torch.empty(q(self.B), dtype=i32, device=dev)
        self.rowlab = torch.empty(q(tot[1]), dtype=i32, device=dev)
        self.collab = torch.empty(q(tot[2]), dtype=i32, device=dev)
        self.trace = torch.zeros((q(tot[3]), 2), dtype=i32, device=dev) if trace else None
        self.snaps = torch.empty(q(tot[4]), dtype=f64, device=dev) if snapshots else None
        self.totals = tot

    def upload(self, packed, non_blocking: bool = False):
        """packed: the B reference-flat tables back to back, [sum cells] fp64 (numpy or a (pinned) CPU tensor)."""
        src = torch.from_numpy(packed) if isinstance(packed, np.ndarray) else packed
        if tuple(src.shape) != (self.totals[0],):
            raise ValueError(f"packed tables must be [{self.totals[0]}] (the sum of the LPs' cells)")
        self.T[: self.totals[0]].copy_(src, non_blocking=non_blocking)

    def run(self, rule: int = N.RULE_REFERENCE):
        """Launch the plan on the resident batch (asynchronous on the current stream)."""
        with torch.cuda.device(self.device):
            N.call("spx_solve_batched_ragged", self.T.data_ptr(), self.plan.plan.ctypes.data, self.d_plan.data_ptr(),
                   rule, self.x.data_ptr(), self.obj.data_ptr(), self.status.data_ptr(), self.npiv.data_ptr(),
                   self.rowlab.data_ptr(), self.collab.data_ptr(), N.ptr(self.trace), N.ptr(self.snaps),
                   torch.cuda.current_stream(self.device).cuda_stream)

    def _packed(self, a, total: int, k: int, name: str) -> np.ndarray:
        """a packed [total] fp64 array; a non-finite entry is a ValueError naming its LP (k: the column of
        ``offsets``, 1 for per-variable arrays, 2 for per-constraint arrays)"""
        a = np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1))
        if a.shape != (total,):
            raise ValueError(f"{name} must be packed [{total}], got {a.shape[0]} entries")
        _check_finite(a, name, self.offsets[:, k])
        return a

    def upload_labels(self, rowlab, collab, non_blocking: bool = False):
        """As ``DeviceBatch.upload_labels``, packed: rowlab [sum m] (as ``x``) and collab [sum n]."""
        rowlab = np.ascontiguousarray(rowlab, dtype=np.int32).reshape(-1)
        collab = np.ascontiguousarray(collab, dtype=np.int32).reshape(-1)
        if rowlab.shape != (self.totals[1],) or collab.shape != (self.totals[2],):
            raise ValueError(f"rowlab must be packed [{self.totals[1]}] and collab [{self.totals[2]}]")
        _check_ragged_labels(rowlab, collab, self.shapes2, self.offsets[:, 1], self.offsets[:, 2])
        self.rowlab[: self.totals[1]].copy_(torch.from_numpy(rowlab), non_blocking=non_blocking)
        self.collab[: self.totals[2]].copy_(torch.from_numpy(collab), non_blocking=non_blocking)

    def change(self, rhs_delta=None, cost_delta=None):
        """As ``DeviceBatch.change``, with rhs_delta packed [sum n] (as ``collab``) and cost_delta packed
        [sum m] (as ``x``) (``spx_warm_change_ragged``)."""
        tot = self.totals
        db = None if rhs_delta is None else self._packed(rhs_delta, tot[2], 2, "rhs_delta")
        dc = None if cost_delta is None else self._packed(cost_delta, tot[1], 1, "cost_delta")
        if self.B == 0 or (db is None and dc is None):
            return
        up = lambda a: None if a is None else torch.from_numpy(a).to(self.device)  # noqa: E731
        d_db, d_dc = up(db), up(dc)
        with torch.cuda.device(self.device):
            N.call("spx_warm_change_ragged", self.T.data_ptr(), self.plan.plan.ctypes.data, self.d_plan.data_ptr(),
                   self.rowlab.data_ptr(), self.collab.data_ptr(), N.ptr(d_db), N.ptr(d_dc),
                   torch.cuda.current_stream(self.device).cuda_stream)

    def resume(self, function, rule: int = N.RULE_REFERENCE):
        """As ``DeviceBatch.resume``, each LP for up to its own cap; function packed [sum m] (as ``x``)
        (``spx_warm_solve_ragged``)."""
        fn = np.ascontiguousarray(np.asarray(function, dtype=np.float64).reshape(-1))
        if fn.shape != (self.totals[1],):
            raise ValueError(f"function must be packed [{self.totals[1]}], got {fn.shape[0]} entries")
        self._function = torch.from_numpy(fn).to(self.device) if self.B else None    # alive until the kernels ran
        with torch.cuda.device(self.device):
            N.call("spx_warm_solve_ragged", self.T.data_ptr(), self.plan.plan.ctypes.data, self.d_plan.data_ptr(),
                   rule, N.ptr(self._function), self.x.data_ptr(), self.obj.data_ptr(), self.status.data_ptr(),
                   self.npiv.data_ptr(), self.rowlab.data_ptr(), self.collab.data_ptr(), N.ptr(self.trace),
                   N.ptr(self.snaps), torch.cuda.current_stream(self.device).cuda_stream)

    def sensitivity(self) -> RaggedSensitivity:
        """Sensitivity report of the final tables the last ``run`` left; synchronises."""
        return _sens_ragged(self.T, self.plan.plan, self.d_plan, self.status, self.rowlab, self.collab, self.B,
                            self.totals, self.shapes, self.offsets, self.device)

    def result(self) -> RaggedResult:
        B, tot = self.B, self.totals
        g = lambda t, k: None if t is None else t[:k].cpu().numpy()  # noqa: E731
        return RaggedResult(g(self.status, B), g(self.npiv, B), g(self.x, tot[1]), g(self.obj, B), g(self.T, tot[0]),
                            g(self.rowlab, tot[1]), g(self.collab, tot[2]), g(self.trace, tot[3]),
                            g(self.snaps, tot[4]), self.shapes.copy(), self.offsets.copy())


def pack_ragged(lps):
    """(constraints, function) pairs -> ([B, 2] shapes, [sum cells] packed reference-flat tables)."""
    from .engine import as_rows_function
    parts, shapes = [], []
    for constraints, function in lps:
        rows, c = as_rows_function(constraints, function)
        shapes.append((rows.shape[0], c.shape[0]))
        parts += [rows.reshape(-1), c]
    packed = np.concatenate(parts) if parts else np.zeros(0)
    return np.asarray(shapes, dtype=np.int64).reshape(-1, 2), np.ascontiguousarray(packed, dtype=np.float64)


def solve_ragged(lps, max_pivots: Union[int, Sequence[int]] = 64, rule: str = "reference", trace: bool = True,
                 snapshots: bool = False, device=None, engine: str = "auto") -> RaggedResult:
    """Solve independent LPs of any mix of shapes in one call.

    lps: a sequence of ``(constraints, function)`` pairs as ``SimplexMethod`` takes them (e.g.
    ``[problem_io.solver_inputs(p) for p in problems]``); max_pivots: an int or one int per LP.
    Each LP's results are, bit for bit, those ``solve_batched`` returns for that LP alone
    (``RaggedResult.lp(k)``).  engine: "auto" (per LP, K4 when it fits one CTA, else K7),
    "auto_global" (as "auto", and K8 above K7's capacity), or "smem", "cluster" or "global"
    for every LP.
    """
    shapes, packed = pack_ragged(lps)
    db = DeviceRaggedBatch(shapes, max_pivots, trace, snapshots, device, engine)
    if db.B:
        db.upload(packed)
        db.run(N.RULES[rule])
    return db.result()


def _uniform_labels(result: BatchResult, fn: str):
    """(rowlab [B, m], collab [B, n], B, n, m) of a host BatchResult given to `fn`, with n, m >= 1"""
    if not isinstance(result, BatchResult):
        raise TypeError(f"{fn}() takes a BatchResult or a RaggedResult, not {type(result).__name__}")
    rowlab = np.ascontiguousarray(result.rowlab, dtype=np.int32)
    collab = np.ascontiguousarray(result.collab, dtype=np.int32)
    if rowlab.ndim != 2 or collab.ndim != 2 or rowlab.shape[0] != collab.shape[0]:
        raise ValueError("result.rowlab must be [B, m] and result.collab [B, n]")
    B, m, n = rowlab.shape[0], rowlab.shape[1], collab.shape[1]
    if n < 1 or m < 1:
        raise ValueError(f"bad shape {n} x {m}")
    return rowlab, collab, B, n, m


def _check_packing(result: RaggedResult, plan: RaggedPlan) -> None:
    """the packed tables, labels and status of a host RaggedResult have the sizes of the LPs of `plan`"""
    tot = plan.totals
    for name, a, k in (("tables", result.tables, tot[0]), ("rowlab", result.rowlab, tot[1]),
                       ("collab", result.collab, tot[2]), ("status", result.status, len(plan.lps))):
        if np.size(a) != k:
            raise ValueError(f"result.{name} has {np.size(a)} entries, the shapes need {k}")


def sensitivity(result: Union[BatchResult, RaggedResult], device=None) -> Union[Sensitivity, RaggedSensitivity]:
    """Sensitivity report of the final tables of a host ``BatchResult`` (``solve_batched``) or ``RaggedResult``
    (``solve_ragged``): uploads the tables, labels and status and runs the report's kernels on ``device``."""
    dev = torch.device(device if device is not None else "cuda")
    up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt).reshape(-1)).to(dev)  # noqa: E731
    if isinstance(result, RaggedResult):
        shapes = np.asarray(result.shapes, dtype=np.int64).reshape(-1, 3)
        B = shapes.shape[0]
        plan = ragged_plan(shapes[:, :2], shapes[:, 2], "auto_global")
        if not np.array_equal(plan.offsets, np.asarray(result.offsets, dtype=np.int64).reshape(-1, 5)):
            raise ValueError("result.offsets are not the packing of result.shapes")
        _check_packing(result, plan)
        if B == 0:
            z = np.zeros
            return RaggedSensitivity(z(0), z(0), z(0), z((0, 2)), z((0, 2)), z(0, bool), shapes.copy(), plan.offsets)
        N.lib()
        return _sens_ragged(up(result.tables, np.float64), plan.plan, torch.from_numpy(plan.plan).to(dev),
                            up(result.status, np.int32), up(result.rowlab, np.int32), up(result.collab, np.int32),
                            B, plan.totals, shapes, plan.offsets, dev)
    rowlab, collab, B, n, m = _uniform_labels(result, "sensitivity")
    if np.shape(result.tables) != (B, n * (m + 1) + m) or np.shape(result.status) != (B,):
        raise ValueError(f"result.tables must be [B, n*(m+1)+m] = [{B}, {n * (m + 1) + m}] and result.status [{B}]")
    if B == 0:
        z = np.zeros
        return Sensitivity(z((0, n)), z((0, n)), z((0, m)), z((0, n, 2)), z((0, m, 2)), z(0, bool))
    N.lib()
    return _sens_uniform(up(result.tables, np.float64), up(result.status, np.int32), up(rowlab, np.int32),
                         up(collab, np.int32), B, n, m, dev)


def _new_values(new, old: np.ndarray, name: str):
    """(new values, delta = new - old) of [B, k] `old`; new None: unchanged, no delta."""
    if new is None:
        return old, None
    new = _per_lp(new, old.shape[0], old.shape[1], name)
    return new, new - old


def _packed_values(new, sizes: np.ndarray, name: str) -> Optional[np.ndarray]:
    """a packed array, or one array per LP -> packed fp64; None stays None"""
    if new is None:
        return None
    if isinstance(new, (list, tuple)) and len(new) == len(sizes) and len(new) and np.ndim(new[0]) == 1:
        for k, (v, s) in enumerate(zip(new, sizes)):
            if np.shape(v) != (int(s),):
                raise ValueError(f"LP {k}: {name} must have {int(s)} entries, got shape {np.shape(v)}")
        new = np.concatenate([np.asarray(v, dtype=np.float64) for v in new])
    new = np.asarray(new, dtype=np.float64).reshape(-1)
    if new.shape != (int(sizes.sum()),):
        raise ValueError(f"{name} must be packed [{int(sizes.sum())}] or one array per LP")
    return new


def resolve(result: Union[BatchResult, RaggedResult], data, rhs=None, cost=None, max_pivots=64,
            rule: str = "reference", trace: bool = True, snapshots: bool = False, device=None,
            engine: str = "auto") -> Union[BatchResult, RaggedResult]:
    """Re-optimise solved LPs after new right-hand sides and/or costs, from their final tables.

    result: a host ``BatchResult`` (``solve_batched``) with data = the [B, cells] tables it was solved from,
    or a ``RaggedResult`` (``solve_ragged``) with data = its ``(constraints, function)`` pairs.  data must hold
    the b and c the final tables currently belong to: to chain, pass the result of an earlier ``resolve`` with
    the tables (or pairs) carrying that call's new b and c, not the original ones, or the deltas are wrong.
    rhs / cost: the new b ([B, n] or [n]) and c ([B, m] or [m]); for a ragged result packed ([sum n],
    [sum m]) or one array per LP.  None keeps the old values; with neither, the LPs simply continue.
    The final tables and labels are uploaded, changed by delta = new - old (``change``) and resumed for up
    to max_pivots more pivots with function = the new costs (``resume``).  Returns the result type given.
    Non-finite deltas, labels that are not a permutation of 0..n+m-1 and shapes that do not match are
    ValueErrors naming the LP.
    """
    if isinstance(result, RaggedResult):
        return _resolve_ragged(result, data, rhs, cost, max_pivots, rule, trace, snapshots, device, engine)
    rowlab, collab, B, n, m = _uniform_labels(result, "resolve")
    cells = n * (m + 1) + m
    tables = np.ascontiguousarray(result.tables, dtype=np.float64)
    data = np.asarray(data, dtype=np.float64)
    if tables.shape != (B, cells) or data.shape != (B, cells):
        raise ValueError(f"result.tables and data must be [B, n*(m+1)+m] = [{B}, {cells}], got "
                         f"{tables.shape} and {data.shape}")
    _check_labels(rowlab, collab)
    new_c, dc = _new_values(cost, data[:, n * (m + 1):], "cost")
    _, db = _new_values(rhs, data[:, : n * (m + 1)].reshape(B, n, m + 1)[:, :, m], "rhs")
    _check_finite(db, "rhs - old rhs")
    _check_finite(dc, "cost - old cost")
    db_ = DeviceBatch(B, n, m, int(max_pivots), trace, snapshots, device, engine)
    if B == 0:
        return _empty_batch(n, m, int(max_pivots), trace, snapshots)
    db_.upload(tables)
    db_.upload_labels(rowlab, collab)
    db_.change(db, dc)
    db_.resume(new_c, N.RULES[rule])
    return db_.result()


def _resolve_ragged(result: RaggedResult, data, rhs, cost, max_pivots, rule, trace, snapshots, device,
                    engine) -> RaggedResult:
    shapes, packed = pack_ragged(data)
    rshapes = np.asarray(result.shapes, dtype=np.int64).reshape(-1, 3)
    if not np.array_equal(shapes, rshapes[:, :2]):
        raise ValueError("data are not the LPs of result (their shapes differ from result.shapes)")
    B = shapes.shape[0]
    plan = ragged_plan(shapes, _caps(max_pivots, B), engine)
    offsets = plan.offsets
    _check_packing(result, plan)
    rowlab = np.ascontiguousarray(result.rowlab, dtype=np.int32).reshape(-1)
    collab = np.ascontiguousarray(result.collab, dtype=np.int32).reshape(-1)
    old_b, old_c = np.empty(int(plan.totals[2])), np.empty(int(plan.totals[1]))
    _check_ragged_labels(rowlab, collab, shapes, offsets[:, 1], offsets[:, 2])
    for k in range(B):
        n, m = (int(v) for v in shapes[k])
        t, xm, xn = (int(v) for v in offsets[k, :3])
        old_b[xn: xn + n] = packed[t: t + n * (m + 1)].reshape(n, m + 1)[:, m]
        old_c[xm: xm + m] = packed[t + n * (m + 1): t + n * (m + 1) + m]
    new_b = _packed_values(rhs, shapes[:, 0], "rhs")
    new_c = _packed_values(cost, shapes[:, 1], "cost")
    deltas = [None if v is None else v - old for v, old in ((new_b, old_b), (new_c, old_c))]
    _check_finite(deltas[0], "rhs - old rhs", offsets[:, 2])
    _check_finite(deltas[1], "cost - old cost", offsets[:, 1])
    db_ = DeviceRaggedBatch(shapes, max_pivots, trace, snapshots, device, engine)
    if B:
        db_.upload(np.ascontiguousarray(result.tables, dtype=np.float64).reshape(-1))
        db_.upload_labels(rowlab, collab)
        db_.change(*deltas)
        db_.resume(old_c if new_c is None else new_c, N.RULES[rule])
    return db_.result()
