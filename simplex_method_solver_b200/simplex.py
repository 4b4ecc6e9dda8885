"""Drop-in replacement for the reference's ``src/simplex.py`` on a B200.

Same names, arguments and error behaviour as /root/reference/src/simplex.py
(``Error`` :4-9, ``Info`` :12-21, ``SimplexMethod`` :24-199) so the reference's
callers — ``MainWindow.compute_solution`` (main.py:308-317) and
``TableWidget.update_from_info`` (table_widget.py:85-134) — run unchanged after
swapping one import.  The tableau lives in HBM; every pick and every pivot is a
hand-written sm_100a kernel reached through the C ABI (include/spx_b200.h).
There is no CPU fallback: constructing a ``SimplexMethod`` without a CUDA
device or without the built library raises.

Differences from the reference, all opt-in or unavoidable:
  * ``max_pivots`` (keyword, default 1,000,000): the reference has no cap and
    loops forever on cycling inputs (e.g. rows [[1,0,3],[2,0,0]], c [-1,0]);
    here ``get_solution`` ends such a run with ``Error("pivot limit reached")``.
  * ``rule="dantzig"`` selects most-negative entering instead of the
    reference's first-negative rule (not reference behaviour; default off).
  * ``constraints`` may be a 2-D fp64 ndarray (used in place for the upload) so
    large tableaus need no list-of-lists; inputs are never mutated.
  * ``solve()`` returns the trace / x / objective without per-pivot snapshots,
    which the reference cannot avoid (it deep-copies the table per pivot, :198).
  * ``engine="cluster"``: ``get_solution()`` runs the whole loop in the batched
    cluster kernel (K7, one thread-block cluster of up to 16 CTAs holds the
    table in shared memory), which writes the per-pivot snapshots itself; for
    LPs above the one-CTA limit of ``engine="warp"``.  ``solve()`` keeps the
    streaming loop, as with ``"warp"``.
  * ``engine="global"``: the same with the global-memory cluster kernel (K8,
    the table stays in HBM and each CTA of the cluster updates its band of
    rows in place), for LPs above K7's capacity up to K8's.  ``solve()`` keeps
    the streaming loop.
  * ``engine="sharded"``: one process per GPU (torchrun); every rank constructs
    the same ``SimplexMethod`` and calls ``solve()`` — the body is split into
    column blocks over the ranks of ``group`` (the default process group) and
    pivoted by the column-sharded fused loop (``parallel.FusedShardedTableau``:
    pricing inside a cooperative kernel with an NVLink peer-memory exchange per
    pivot).  b, labels, trace, x and the objective are replicated, so
    ``solve()``, ``find_optimum()``, ``f()``, ``row``/``column`` behave as on one
    GPU; the step API and ``get_solution()``/``table`` (a snapshot per pivot of a
    table no rank holds) raise ``NotImplementedError``.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _native as N
from .batched import DeviceBatch, Sensitivity, _SensOut, kernel_for
from .engine import DeviceTableau, Solution, as_rows_function

CAP_TEXT = "pivot limit reached"


class Error:
    """simplex.py:4-9"""

    def __init__(self, error_string):
        self.error_string = error_string

    def __str__(self):
        return self.error_string


class Info:
    """Per-iteration snapshot handed to the GUI widgets (simplex.py:12-21)."""

    def __init__(self, row, column, table, i, j, x1, x2, optimum):
        self.row = list(row)
        self.column = list(column)
        self.table = [list(r) for r in table] if table is not None else None
        self.i = i
        self.j = j
        self.x1 = x1
        self.x2 = x2
        self.optimum = optimum


def _ragged(flat: np.ndarray, n: int, m: int):
    """reference-flat -> the reference's list of lists (n rows of m+1, f row of m)."""
    body = flat[: n * (m + 1)].reshape(n, m + 1).tolist()
    body.append(flat[n * (m + 1):].tolist())
    return body


class SimplexMethod:
    SHARDED_TRACE_MAX = 1 << 22           # pivots a sharded solve can trace (8 B each)

    def __init__(self, constraints, function, *, max_pivots: int = 1_000_000,
                 rule: str = "reference", device=None, engine: str = "auto", group=None):
        rows, c = as_rows_function(constraints, function)
        self.n = rows.shape[0]                               # :26
        self.m = rows.shape[1] - 1                           # :27
        self.invalid_index = 1 + max(self.n, self.m)         # :28
        self.function = function                             # :29 (same object, never mutated)
        self.row = ['x' + str(k) for k in range(1, self.m + 1)] + ['-b']      # :30,:32
        self.column = ['y' + str(k) for k in range(1, self.n + 1)] + ['f']    # :31,:33
        if rule not in N.RULES:
            raise ValueError(f"unknown rule {rule!r}")
        if engine not in ("auto", "warp", "stream", "sharded", "cluster", "global"):
            raise ValueError(f"unknown engine {engine!r}")
        self._rule = N.RULES[rule]
        self._engine = engine
        self._max_pivots = int(max_pivots)
        self._c = c
        self._npiv = 0
        self._table_cache = None
        self._sh = None
        if engine == "sharded":
            self._dev = None
            self._open_sharded(rows, c, device, group)
            return
        self._dev = DeviceTableau(self.n, self.m, device=device)
        self._dev.load(rows, c)

    # ------------------------------------------------------------------ column-sharded engine
    def _open_sharded(self, rows, c, device, group):
        import torch.distributed as dist
        from .parallel import FusedShardedTableau
        if dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(group), dist.get_world_size(group)
        else:
            rank, world = 0, 1
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self._trace_cap = min(self._max_pivots, self.SHARDED_TRACE_MAX)
        self._sh = FusedShardedTableau(self.n, self.m, rank, world, device, trace_capacity=self._trace_cap + 64,
                                       group=group, rule=self._rule)
        self._sh.load(rows, c, max_pivots=self._max_pivots)
        self._fn_dev = torch.from_numpy(np.ascontiguousarray(c, dtype=np.float64)).to(self._sh.device)
        self._x_dev = torch.zeros(max(self.m, 1), dtype=torch.float64, device=self._sh.device)
        self._obj_dev = torch.zeros(2, dtype=torch.float64, device=self._sh.device)

    def _not_sharded(self, what):
        if self._sh is not None:
            raise NotImplementedError(f"{what} is not available with engine='sharded' (no rank holds the whole table); "
                                      "use solve(), find_optimum(), f()")

    def _solve_sharded(self, cap, chunk):
        sh = self._sh
        if self._npiv + cap > self._trace_cap:
            raise ValueError(f"engine='sharded': {self._npiv + cap} pivots exceed the trace capacity {self._trace_cap} "
                             "fixed at construction (max_pivots)")
        total = self._npiv + cap
        st = sh.read_state()                                 # (synchronises; keeps reserved[0] = the current buffer)
        if int(st.max_pivots) != total or st.status == N.CAP:
            st.max_pivots = total
            if st.status == N.CAP:
                st.status = N.PIVOT
            sh.state.copy_(torch.from_numpy(np.frombuffer(bytes(st), dtype=np.int64).copy()))
        status, npiv = sh.solve(total, check_every=max(int(chunk), 1))
        self._npiv = int(npiv)
        with torch.cuda.device(sh.device):
            N.call("spx_extract", sh.b_current().data_ptr(), self.n, self.m, sh.collab.data_ptr(), self._fn_dev.data_ptr(),
                   self._x_dev.data_ptr(), self._obj_dev.data_ptr(), torch.cuda.current_stream(sh.device).cuda_stream)
        x = self._x_dev[: self.m].cpu().numpy()
        obj = self._obj_dev.cpu().numpy()
        rl, cl = sh.rowlab.cpu().numpy(), sh.collab[: self.n].cpu().numpy()
        sol = Solution(int(status), self._npiv, sh.trace[: self._npiv].cpu().numpy(), x, float(obj[0]), float(obj[1]), rl, cl)
        self._labels_from_codes(rl, cl)
        return sol

    def close(self):
        """engine='sharded': release the peer-memory mappings (collective: every rank calls it)."""
        if self._sh is not None:
            self._sh.close()
            self._sh = None

    # ------------------------------------------------------------------ views
    @property
    def table(self):
        """Current tableau as the reference's list of lists (:36-39), read back from HBM."""
        self._not_sharded("table")
        if self._table_cache is None:
            self._table_cache = _ragged(self._dev.export_flat(self._npiv), self.n, self.m)
        return self._table_cache

    def print_table(self):                                   # :41-46
        print("\t", end='')
        print("\t".join(self.row))
        tab = self.table
        for k in range(self.n + 1):
            print(self.column[k], end='\t')
            print("\t".join(str(round(v, 6)) for v in tab[k]))

    def f(self, x1, x2):                                     # :48-49
        return self.function[0] * x1 + self.function[1] * x2

    def find_optimum(self):                                  # :51-68
        b = None
        out = []
        for name in ('x1', 'x2'):
            if name in self.column:
                if b is None:
                    b = (self._sh.b_current().cpu().numpy() if self._sh is not None else self._dev.b_host(self._npiv))
                out.append(float(b[self.column.index(name)]))
            else:
                out.append(0)
        return out[0], out[1]

    # ------------------------------------------------------------------ K1+K2
    def _pick_state(self):
        self._not_sharded("the step API (pick_element / recalculate_matrix)")
        self._dev.pick(self._npiv, self._rule, sticky=False)
        st = self._dev.read_state()
        if st.status == N.CAP:
            # the cap belongs to solve()/get_solution(); the reference's step API has none
            st.max_pivots = 1 << 62
            st.status = N.PIVOT
            self._dev.write_state(st)
            self._dev.pick(self._npiv, self._rule, sticky=False)
            st = self._dev.read_state()
        return st

    def pick_element(self):                                  # :70-141
        st = self._pick_state()
        if st.status == N.PIVOT:
            return True, int(st.r), int(st.c), float(st.p)
        if st.status == N.OPTIMAL:
            x1, x2 = self.find_optimum()
            return False, x1, x2, self.f(x1, x2)
        raise ValueError(N.ERROR_TEXT[st.status])

    # ------------------------------------------------------------------ K3
    def _swap_labels(self, r, c):                            # :152
        self.row[c], self.column[r] = self.column[r], self.row[c]

    def recalculate_matrix(self):                            # :143-177
        st = self._pick_state()                              # the reference picks again here (:144)
        if st.status == N.OPTIMAL:
            return
        if st.status != N.PIVOT:
            raise ValueError(N.ERROR_TEXT[st.status])
        self._dev.update(self._npiv)
        self._npiv += 1
        self._swap_labels(int(st.r), int(st.c))
        self._table_cache = None

    # ------------------------------------------------------------------ loops
    def _use_warp(self):
        if self._engine == "stream":
            return False
        if self._engine in ("cluster", "global"):
            kernel_for(self.n, self.m, self._engine)     # ValueError above the engine's capacity
            return True
        cells = self.n * (self.m + 1) + self.m
        L = N.load()
        fits = bool(L.spx_batched_fits(self.n, self.m))
        if self._engine == "warp" and not fits:
            raise ValueError("engine='warp' needs the LP to fit shared memory")
        return fits and (self._engine == "warp" or cells <= 2048)

    def _xy(self, column, flat):
        """find_optimum() evaluated on a snapshot."""
        w1 = self.m + 1
        vals = []
        for name in ('x1', 'x2'):
            vals.append(float(flat[column.index(name) * w1 + self.m]) if name in column else 0)
        return vals[0], vals[1]

    def get_solution(self, snapshots: bool = True):          # :179-199
        """list of Info (one per iteration), ending in Error on failure.

        snapshots=False keeps Info.table only on the last Info (large tableaus).
        """
        self._not_sharded("get_solution()")
        result = [Info(self.row, self.column, self.table if snapshots else None,
                       None, None, 0, 0, 0)]                 # :181
        budget = self._max_pivots
        final_status = None
        if self._use_warp():
            final_status = self._solve_warp(result, budget, snapshots)
        else:
            final_status = self._solve_stream(result, budget, snapshots)
        if not snapshots and not isinstance(result[-1], Error):
            result[-1].table = [list(r) for r in self.table]
        if final_status in N.ERROR_TEXT:
            result.append(Error(N.ERROR_TEXT[final_status]))     # :187-189
        elif final_status == N.CAP:
            result.append(Error(CAP_TEXT))
        return result

    def _append_info(self, result, r, c, flat, snapshots):
        result[-1].i, result[-1].j = r, c                    # :194-195
        self._swap_labels(r, c)
        x1, x2 = self._xy(self.column, flat)
        result.append(Info(self.row, self.column,
                           _ragged(flat, self.n, self.m) if snapshots else None,
                           None, None, x1, x2, self.f(x1, x2)))   # :197-198

    def _solve_warp(self, result, budget, snapshots):
        """Whole loop in one batched kernel launch (K4, K7 with engine="cluster", K8 with engine="global")
        per round of `cap` pivots."""
        n, m = self.n, self.m
        engine = self._engine if self._engine in ("cluster", "global") else "smem"
        # rounds of up to `limit` pivots, so that one round's snapshots, (cap + 1) * cells doubles, stay under ~256 MB:
        # K4 and K7 tables are small enough for rounds of 64 and more; a K8 table may allow fewer, down to one pivot
        # (two snapshot tables) for the largest
        cells = n * (m + 1) + m
        limit = (256 << 20) // (8 * cells)
        limit = max(1, limit - 1) if engine == "global" else max(64, limit)
        cap = min(64, limit)
        while True:
            cap = min(cap, max(budget, 0))
            db = DeviceBatch(1, n, m, max_pivots=cap, trace=True, snapshots=True,
                             device=self._dev.device, engine=engine)
            self._dev.export_device_flat(self._npiv, db.T[0])
            db.run(self._rule)
            res = db.result()
            k = int(res.npiv[0])
            status = int(res.status[0])
            for q in range(k):
                r, c = int(res.trace[0, q, 0]), int(res.trace[0, q, 1])
                self._append_info(result, r, c, res.snaps[0, q + 1], snapshots)
            # keep the streaming state coherent: final table -> buffer (npiv+k)&1, labels, counter
            self._npiv += k
            self._dev.load_device_flat(db.T[0], self._dev.cur(self._npiv))
            self._push_labels()
            self._table_cache = None
            budget -= k
            if status != N.CAP or budget <= 0:
                return status
            cap = min(cap * 4, limit)                        # grow the round up to the bound above

    def _push_labels(self):
        code = lambda s: int(s[1:]) - 1 if s[0] == 'x' else self.m + int(s[1:]) - 1  # noqa: E731
        rl = np.asarray([code(s) for s in self.row[:-1]], dtype=np.int32)
        cl = np.asarray([code(s) for s in self.column[:-1]], dtype=np.int32)
        self._dev.rowlab.copy_(torch.from_numpy(rl))
        self._dev.collab[: self.n].copy_(torch.from_numpy(cl))
        st = self._dev.read_state()
        st.npiv = self._npiv
        st.status = N.PIVOT
        st.hint_tag[0] = st.hint_tag[1] = -1
        self._dev.write_state(st)

    def _solve_stream(self, result, budget, snapshots):
        """pick + update kernels per pivot; one state read-back per pivot (snapshots need it)."""
        while True:
            st = self._pick_state()
            if st.status != N.PIVOT:
                return st.status
            if budget <= 0:
                return N.CAP
            self._dev.update(self._npiv)
            self._npiv += 1
            budget -= 1
            self._table_cache = None
            flat = self._dev.export_flat(self._npiv) if snapshots else None
            if flat is None:
                # only the b column is needed for x1/x2
                b = self._dev.b_host(self._npiv)
                flat = np.zeros(self.n * (self.m + 1) + self.m)
                flat[self.m: self.n * (self.m + 1): self.m + 1] = b
            self._append_info(result, int(st.r), int(st.c), flat, snapshots)

    def solve(self, max_pivots=None, chunk: int = 64, trace: bool = True, lookahead=None) -> Solution:
        """Device-side loop without snapshots: status, pivot trace, x[0..m), objective.

        Continues from the current table; the pivot loop runs as pre-enqueued
        pick+update kernel pairs with one host read-back per `chunk` pivots.
        """
        cap = self._max_pivots if max_pivots is None else int(max_pivots)
        if self._sh is not None:
            return self._solve_sharded(cap, chunk if chunk != 64 else 4096)
        dev = self._dev
        start = self._npiv
        if trace:
            need = start + cap
            if dev.trace is None or dev.trace_capacity < need:
                old = dev.trace
                dev.trace = torch.zeros((need, 2), dtype=torch.int32, device=dev.device)
                if old is not None and start > 0:
                    keep = min(start, old.shape[0])     # step-API pivots beyond the old capacity are not traced
                    dev.trace[:keep].copy_(old[:keep])
                dev.trace_capacity = need
        else:
            dev.trace = None
            dev.trace_capacity = 0
        st = dev.read_state()
        st.max_pivots = start + cap
        if st.status == N.CAP:
            st.status = N.PIVOT
        dev.write_state(st)
        status, npiv = dev.solve(self._rule, chunk=chunk, lookahead=lookahead)
        self._npiv = int(npiv)
        self._table_cache = None
        sol = dev.solution(status, self._npiv)
        self._labels_from_codes(sol.rowlab, sol.collab)
        return sol

    def sensitivity(self) -> Sensitivity:
        """Sensitivity report of the current table, which must be optimal: after ``solve()``, ``get_solution()``
        or step-API pivots.  Arrays without the batch axis: dual, slack [n], reduced_cost [m], rhs_range [n, 2],
        cost_range [m, 2]; ``optimal`` is True.  ValueError when the current table is not optimal."""
        self._not_sharded("sensitivity()")
        dev, n, m = self._dev, self.n, self.m
        c = dev.cur(self._npiv)
        out = _SensOut(n, m, dev.device)
        optimal = ctypes.c_int32(0)
        dev._call("spx_sensitivity_split", dev.A[c].data_ptr(), dev.b[c].data_ptr(), n, m, dev.ld,
                  dev.rowlab.data_ptr(), dev.collab.data_ptr(), *out.ptrs(), ctypes.byref(optimal))
        if not optimal.value:
            raise ValueError("sensitivity() needs an optimal table: the current table has a negative b or f cell "
                             "(solve the LP to optimality first)")
        dual, slack, rc, rr, cr = out.host()
        return Sensitivity(dual, slack, rc, rr.reshape(n, 2), cr.reshape(m, 2), True)

    def _labels_from_codes(self, rowlab, collab):
        name = lambda v: f"x{v + 1}" if v < self.m else f"y{v - self.m + 1}"  # noqa: E731
        self.row = [name(int(v)) for v in rowlab] + ['-b']
        self.column = [name(int(v)) for v in collab] + ['f']
