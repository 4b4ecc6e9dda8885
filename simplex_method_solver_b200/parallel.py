"""Multi-GPU paths: one process per GPU, ``torch.distributed`` for the plumbing.

Two partitionings, the two places where the pivot loop shards naturally
(SURVEY.md §8e):

* **Batches of independent small LPs** — contiguous split of the batch, no
  data-path collective (``shard_range`` + ``solve_batched_sharded``; for LPs of
  mixed shapes ``cells_range`` + ``solve_ragged_sharded``, balanced by cells).

* **Column-sharded large tableau** — rank g owns a contiguous block of body
  columns as its own split matrix; the b column, labels and the 128-byte solver
  state are replicated.  One exchange per pivot: every rank packs
  ``[key | its candidate entering column]`` (K1 local half) and a single
  all-gather over NCCL/NVLink delivers all candidates everywhere; each rank
  then takes the lexicographic-min key (K1 global half), runs the ratio test on
  the winning column with its replica of b (K2, redundantly — bit-identical on
  all ranks) and updates its own columns (K3).  No host round trip, no
  data-dependent broadcast root.  The pivot trace equals the single-GPU trace
  exactly (tests/test_sharded_gloo.py on CPU with gloo; bench.py on GPUs).

  With ``lookahead=True`` the exchange leaves the critical path: pivot k+1 is
  priced from table k (the look-ahead kernels of csrc/spx_pick.cu compute the
  next b column, the next f / phase-1 row and the next entering column with the
  update's own arithmetic), so candidate -> all-gather -> select run on a
  high-priority side stream WHILE update k streams on the main stream; state and
  colbuf are double-buffered and the two streams join once per pivot.

The kernels are reached through ``ShardOps``; the product implementation
(``CudaShardOps``) calls the C ABI.  Tests inject a CPU stand-in to exercise
this file's collective logic under gloo without a GPU.
"""
from __future__ import annotations

import contextlib
import ctypes
import os
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _native as N

MSG_HEADER = 4     # doubles: [key_hi, key_lo, r_phase1, reserved] (csrc/spx_pick.cu)
TILE_COLS = 512    # column tile of the update kernel (csrc/spx_update.cu)


def shard_range(total: int, rank: int, world: int):
    """Contiguous split of `total` units: (start, count) of `rank`; sizes differ by at most 1."""
    base, rem = divmod(int(total), int(world))
    start = rank * base + min(rank, rem)
    return start, base + (1 if rank < rem else 0)


def column_block(m: int, rank: int, world: int, align: int = TILE_COLS):
    """Column block of `rank`: contiguous, boundaries on multiples of `align` (whole update tiles)."""
    tiles = -(-int(m) // align)
    t0, tc = shard_range(tiles, rank, world)
    col0 = min(t0 * align, m)
    col1 = min((t0 + tc) * align, m)
    return col0, col1 - col0


def msg_doubles(n: int) -> int:
    return (MSG_HEADER + n + 1 + 15) // 16 * 16


def _p(x):
    """Device pointer of a tensor, or the integer address itself."""
    return x if isinstance(x, int) or x is None else x.data_ptr()


class PeerMailboxes:
    """Every rank's mailbox mapped into this process (CUDA IPC): the NVLink exchange of the sharded flow.

    Layout per rank (csrc/spx_shard.cu): gathered[2][world][msg] | flags[2][world].  The local box is
    cudaMalloc'ed by the library (exportable), the peers' boxes are opened from handles exchanged
    once through torch.distributed — plumbing only; the per-pivot exchange is spx_peer_push.
    """

    def __init__(self, n: int, rank: int, world: int, device, group=None, local_only_ptrs=None):
        L = N.lib()
        self.n, self.rank, self.world = int(n), int(rank), int(world)
        self.device = torch.device(device)
        self.msgd = int(L.spx_shard_msg_doubles(self.n))
        self.bytes = int(L.spx_mailbox_bytes(self.n, self.world))
        self.flags_offset = (2 * self.world * self.msgd * 8 + 127) // 128 * 128
        self._opened = []
        with torch.cuda.device(self.device):
            local = ctypes.c_void_p()
            N.call("spx_device_alloc", ctypes.byref(local), self.bytes)
            self.local = int(local.value)
            ptrs = [None] * self.world
            ptrs[self.rank] = self.local
            if local_only_ptrs is not None:            # several ranks emulated inside one process (tests)
                self._shared = local_only_ptrs
                local_only_ptrs[self.rank] = self.local
                self.ptrs = None
                return
            if self.world > 1:
                hb = int(L.spx_ipc_handle_bytes())
                buf = (ctypes.c_ubyte * hb)()
                N.call("spx_ipc_export", self.local, buf)
                handles = [None] * self.world
                dist.all_gather_object(handles, bytes(buf), group=group)
                for g in range(self.world):
                    if g == self.rank:
                        continue
                    hbuf = (ctypes.c_ubyte * hb).from_buffer_copy(handles[g])
                    q = ctypes.c_void_p()
                    N.call("spx_ipc_import", hbuf, ctypes.byref(q))
                    ptrs[g] = int(q.value)
                    self._opened.append(int(q.value))
            self.ptrs = (ctypes.c_void_p * self.world)(*ptrs)

    def finalize_shared(self):
        """Emulation only: call once every emulated rank has allocated its box."""
        self.ptrs = (ctypes.c_void_p * self.world)(*self._shared)

    def gathered_ptr(self, parity: int) -> int:
        return self.local + parity * self.world * self.msgd * 8

    def flags_ptr(self, parity: int) -> int:
        return self.local + self.flags_offset + parity * self.world * 8

    def close(self, group=None):
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            for q in self._opened:
                N.call("spx_ipc_close", q)
            self._opened = []
            if self.world > 1 and dist.is_initialized() and self.ptrs is not None and getattr(self, "_shared", None) is None:
                dist.barrier(group=group)              # nobody frees a box a peer still has mapped
            if self.local:
                N.call("spx_device_free", self.local)
                self.local = 0


class CudaShardOps:
    """The three per-pivot kernels of the sharded flow, through the C ABI."""

    def __init__(self, device):
        N.lib()
        self.device = torch.device(device)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def import_shard(self, rows, function, A, b, n, m, col0, m_loc, ld):
        N.call("spx_import_shard", rows.ctypes.data, function.ctypes.data, A.data_ptr(), b.data_ptr(),
               n, m, col0, m_loc, ld, self._stream())
        torch.cuda.current_stream(self.device).synchronize()

    def init_state(self, state, rowlab, collab, n, m, max_pivots):
        N.call("spx_init_state", state.data_ptr(), rowlab.data_ptr(), collab.data_ptr(), n, m,
               max_pivots, self._stream())

    def candidate(self, A, b, n, m_loc, ld, col0, rule, state, send):
        N.call("spx_shard_candidate", A.data_ptr(), b.data_ptr(), n, m_loc, ld, col0, rule, 1,
               state.data_ptr(), send.data_ptr(), self._stream())

    def select(self, gathered, world, b, n, rule, state, colbuf, flags=None, seq=0):
        N.call("spx_shard_select", _p(gathered), world, b.data_ptr(), n, rule, 1,
               state.data_ptr(), colbuf.data_ptr(), flags, seq, self._stream())

    def push(self, send, n, rank, world, parity, seq, ptrs):
        N.call("spx_peer_push", send.data_ptr(), n, rank, world, parity, seq, ptrs, self._stream())

    def update(self, Ain, Aout, bin_, bout, n, m_loc, ld, col0, state, colbuf, rowlab, collab, trace,
               ahead=False):
        N.call("spx_shard_update", Ain.data_ptr(), Aout.data_ptr(), bin_.data_ptr(), bout.data_ptr(),
               n, m_loc, ld, col0, state.data_ptr(), colbuf.data_ptr(), rowlab.data_ptr(),
               collab.data_ptr(), N.ptr(trace), int(ahead), self._stream())

    def ahead_candidate(self, A, bin_, bout, n, m_loc, ld, col0, rule, state, colbuf, send):
        N.call("spx_ahead_candidate", A.data_ptr(), bin_.data_ptr(), bout.data_ptr(), n, m_loc, ld, col0,
               rule, state.data_ptr(), colbuf.data_ptr(), send.data_ptr(), self._stream())

    def ahead_select(self, gathered, world, bnext, n, state_cur, state_next, colbuf_next, flags=None, seq=0):
        N.call("spx_ahead_select", _p(gathered), world, bnext.data_ptr(), n, state_cur.data_ptr(),
               state_next.data_ptr(), colbuf_next.data_ptr(), flags, seq, self._stream())


class ShardedTableau:
    """One rank's share of a column-sharded tableau plus the replicated pieces."""

    def __init__(self, n: int, m: int, rank: int, world: int, device, trace_capacity: int = 0,
                 group=None, ops=None, rule: int = N.RULE_REFERENCE, lookahead: bool = False,
                 mailboxes: Optional["PeerMailboxes"] = None):
        self.n, self.m, self.rank, self.world = int(n), int(m), int(rank), int(world)
        self.device = torch.device(device)
        self.group = group
        self.rule = rule
        self.lookahead = bool(lookahead)
        self.mailboxes = mailboxes     # None: the exchange is a torch.distributed all-gather
        self.seq = 0                   # exchanges issued (mailbox mode); parity = seq & 1
        self.ops = ops if ops is not None else CudaShardOps(self.device)
        self.col0, self.m_loc = column_block(self.m, self.rank, self.world)
        self.ld = max(16, (self.m_loc + 15) // 16 * 16)
        self.nb = (self.n + 15) // 16 * 16
        dev = self.device
        f64, i32 = torch.float64, torch.int32
        self.A = torch.zeros((2, self.n + 1, self.ld), dtype=f64, device=dev)
        self.b = torch.zeros((2, self.nb), dtype=f64, device=dev)
        self.colbuf = torch.zeros((self.n + 1 + 63) // 64 * 64 + 64, dtype=f64, device=dev)
        self.state = torch.zeros(ctypes.sizeof(N.SpxState) // 8, dtype=torch.int64, device=dev)
        self.rowlab = torch.zeros(self.m, dtype=i32, device=dev)
        self.collab = torch.zeros(max(self.n, 1), dtype=i32, device=dev)
        self.msgd = msg_doubles(self.n)
        self.send = torch.zeros(self.msgd, dtype=f64, device=dev)
        self.gathered = torch.zeros((self.world, self.msgd), dtype=f64, device=dev)
        self.trace = torch.zeros((trace_capacity, 2), dtype=i32, device=dev) if trace_capacity > 0 else None
        self.npiv_enqueued = 0
        # look-ahead: second state / colbuf, the side stream and the fork/join events
        self.states = [self.state, torch.zeros_like(self.state)]
        self.colbufs = [self.colbuf, torch.zeros_like(self.colbuf)]
        self.si = 0                  # which of the two holds the decision for the current table
        self.priced = False
        self.side = self.fork = self.join = None
        if self.lookahead and self.device.type == "cuda":
            self.side = torch.cuda.Stream(device=self.device, priority=-1)
            self.fork, self.join = torch.cuda.Event(), torch.cuda.Event()

    def load(self, rows: np.ndarray, function: np.ndarray, max_pivots: int):
        """Every rank reads its own column block (and the whole b column) of the same host table."""
        assert rows.shape == (self.n, self.m + 1) and rows.dtype == np.float64 and rows.flags.c_contiguous
        self.ops.import_shard(rows, np.ascontiguousarray(function, dtype=np.float64), self.A[0], self.b[0],
                              self.n, self.m, self.col0, self.m_loc, self.ld)
        self.ops.init_state(self.state, self.rowlab, self.collab, self.n, self.m, int(max_pivots))
        self.npiv_enqueued = 0
        self.si, self.priced = 0, False

    def load_local(self, block: np.ndarray, function_block: np.ndarray, max_pivots: int):
        """Upload this rank's OWN packed block: `block` is [n, m_loc + 1] = this rank's columns followed by
        the b column (e.g. a view of pinned host memory), `function_block` its m_loc objective entries."""
        assert block.shape == (self.n, self.m_loc + 1) and block.dtype == np.float64 and block.flags.c_contiguous
        fb = np.ascontiguousarray(function_block, dtype=np.float64)
        assert fb.shape == (self.m_loc,)
        # the packed block's own width is its source pitch: m_loc columns + the b column (m_loc == 0: b alone)
        self.ops.import_shard(block, fb, self.A[0], self.b[0], self.n, self.m_loc, 0, self.m_loc, self.ld)
        self.ops.init_state(self.state, self.rowlab, self.collab, self.n, self.m, int(max_pivots))
        self.npiv_enqueued = 0
        self.si, self.priced = 0, False

    def _all_gather(self):
        if self.world > 1:
            dist.all_gather_into_tensor(self.gathered.view(-1), self.send, group=self.group)
        else:
            self.gathered[0].copy_(self.send)

    def _on_side(self):
        """Context that makes the side stream current (no-op for the CPU stand-in)."""
        return torch.cuda.stream(self.side) if self.side is not None else contextlib.nullcontext()

    # A pivot is three phases so that tests can emulate several ranks in one process by running
    # each phase for every rank in lockstep: local half -> exchange -> global half + update.
    def phase_local(self):
        cur = self.npiv_enqueued & 1
        if not self.lookahead:
            self.ops.candidate(self.A[cur], self.b[cur], self.n, self.m_loc, self.ld, self.col0, self.rule,
                               self.state, self.send)
            return
        S, C, si = self.states, self.colbufs, self.si
        if self.side is not None:
            self.fork.record(torch.cuda.current_stream(self.device))
            self.side.wait_event(self.fork)
        with self._on_side():
            self.ops.ahead_candidate(self.A[cur], self.b[cur], self.b[cur ^ 1], self.n, self.m_loc, self.ld,
                                     self.col0, self.rule, S[si], C[si], self.send)

    def _exchange(self, gather=None):
        if self.mailboxes is not None:       # NVLink peer stores + flags, no collective
            self.seq += 1
            self.ops.push(self.send, self.n, self.rank, self.world, self.seq & 1, self.seq, self.mailboxes.ptrs)
        else:
            (gather or self._all_gather)()

    def _gathered_and_flags(self):
        if self.mailboxes is None:
            return self.gathered, None, 0
        par = self.seq & 1
        return self.mailboxes.gathered_ptr(par), self.mailboxes.flags_ptr(par), self.seq

    def phase_exchange(self, gather=None):
        with (self._on_side() if self.lookahead else contextlib.nullcontext()):
            self._exchange(gather)

    def phase_global(self):
        cur = self.npiv_enqueued & 1
        gathered, flags, seq = self._gathered_and_flags()
        if not self.lookahead:
            self.ops.select(gathered, self.world, self.b[cur], self.n, self.rule, self.state, self.colbuf,
                            flags, seq)
            self.ops.update(self.A[cur], self.A[cur ^ 1], self.b[cur], self.b[cur ^ 1], self.n, self.m_loc,
                            self.ld, self.col0, self.state, self.colbuf, self.rowlab, self.collab, self.trace)
        else:
            S, C, si = self.states, self.colbufs, self.si
            with self._on_side():
                self.ops.ahead_select(gathered, self.world, self.b[cur ^ 1], self.n, S[si], S[si ^ 1],
                                      C[si ^ 1], flags, seq)
                if self.side is not None:
                    self.join.record(self.side)
            # the streaming update of pivot k: main stream, concurrent with the pricing above
            self.ops.update(self.A[cur], self.A[cur ^ 1], self.b[cur], self.b[cur ^ 1], self.n, self.m_loc,
                            self.ld, self.col0, S[si], C[si], self.rowlab, self.collab, self.trace, ahead=True)
            if self.side is not None:
                torch.cuda.current_stream(self.device).wait_event(self.join)
            self.si ^= 1
        self.npiv_enqueued += 1

    def first_pick(self, gather=None):
        """Look-ahead only: the decision for the current table from a classic pick (once per load)."""
        if not self.lookahead or self.priced:
            return
        cur, si = self.npiv_enqueued & 1, self.si
        self.ops.candidate(self.A[cur], self.b[cur], self.n, self.m_loc, self.ld, self.col0, self.rule,
                           self.states[si], self.send)
        self._exchange(gather)
        gathered, flags, seq = self._gathered_and_flags()
        self.ops.select(gathered, self.world, self.b[cur], self.n, self.rule, self.states[si],
                        self.colbufs[si], flags, seq)
        self.priced = True

    def step(self):
        """One pivot.  Classic: candidate -> all-gather -> select -> update on one stream.
        Look-ahead: update k on the main stream while candidate -> all-gather -> select price pivot
        k+1 from the same old table on the side stream; the streams join once per pivot."""
        self.first_pick()
        self.phase_local()
        self.phase_exchange()
        self.phase_global()

    def run(self, pivots: int, check_every: int = 0):
        """Enqueue `pivots` pivots; with check_every > 0 stop early on a terminal status.

        Buffer parity follows the number of pivots actually applied, so after an
        early stop the enqueue counter is re-synchronised from the device state.
        """
        done = 0
        while done < pivots:
            k = pivots - done if check_every <= 0 else min(check_every, pivots - done)
            for _ in range(k):
                self.step()
            done += k
            if check_every > 0:
                st = self.read_state()
                if st.status != N.PIVOT:
                    self.npiv_enqueued = int(st.npiv)
                    return st
        return None

    def read_state(self) -> N.SpxState:
        host = self.states[self.si if self.lookahead else 0].cpu().numpy()
        st = N.SpxState.from_buffer_copy(host.tobytes())
        return st

    def solve(self, max_pivots: int, check_every: int = 64):
        """Pivot to a terminal status; returns (status, npiv).

        The cap lives in the device state (set by load()): once npiv reaches it the next
        select reports SPX_CAP — or the real ending if the table is terminal at that point —
        exactly as the single-GPU pick does, and every later kernel of the chunk is a no-op.
        `max_pivots` only bounds the host loop against a state that was loaded with a larger cap.
        """
        while True:
            st = self.run(check_every, check_every=check_every)
            if st is None:
                st = self.read_state()
            if st.status == N.PIVOT and st.npiv >= st.max_pivots:
                self.npiv_enqueued = int(st.npiv)
                self.step()                      # the select of this step reports the ending
                st = self.read_state()
            if st.status != N.PIVOT or st.npiv >= max_pivots:
                self.npiv_enqueued = int(st.npiv)
                return int(st.status), int(st.npiv)

    def sync(self) -> N.SpxState:
        """Read the device state and re-derive the ping-pong parity from the pivots applied."""
        st = self.read_state()
        self.npiv_enqueued = int(st.npiv)
        return st

    def local_body(self) -> torch.Tensor:
        """This rank's current columns [(n+1), m_loc] (row n = f)."""
        self.sync()
        return self.A[self.npiv_enqueued & 1, :, : self.m_loc]

    def b_current(self) -> torch.Tensor:
        self.sync()
        return self.b[self.npiv_enqueued & 1, : self.n]


class PeerRegion:
    """`nbytes` of zeroed device memory on every rank, each rank's block mapped into every process
    (cudaMalloc + CUDA IPC; handles exchanged once through torch.distributed)."""

    def __init__(self, nbytes: int, rank: int, world: int, device, group=None):
        L = N.lib()
        self.rank, self.world, self.device, self.group = int(rank), int(world), torch.device(device), group
        self._opened = []
        with torch.cuda.device(self.device):
            local = ctypes.c_void_p()
            N.call("spx_device_alloc", ctypes.byref(local), int(nbytes))
            self.local = int(local.value)
            ptrs = [None] * self.world
            ptrs[self.rank] = self.local
            if self.world > 1:
                hb = int(L.spx_ipc_handle_bytes())
                buf = (ctypes.c_ubyte * hb)()
                N.call("spx_ipc_export", self.local, buf)
                handles = [None] * self.world
                dist.all_gather_object(handles, bytes(buf), group=group)
                for g in range(self.world):
                    if g == self.rank:
                        continue
                    q = ctypes.c_void_p()
                    N.call("spx_ipc_import", (ctypes.c_ubyte * hb).from_buffer_copy(handles[g]), ctypes.byref(q))
                    ptrs[g] = int(q.value)
                    self._opened.append(int(q.value))
            self.ptrs = (ctypes.c_void_p * self.world)(*ptrs)

    def close(self):
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            for q in self._opened:
                N.call("spx_ipc_close", q)
            self._opened = []
            if self.world > 1 and dist.is_initialized():
                dist.barrier(group=self.group)           # nobody frees a block a peer still has mapped
            if self.local:
                N.call("spx_device_free", self.local)
                self.local = 0


def choose_price_engine(lookahead, world: int, forced: str = "", persistent_from: int = 0) -> int:
    """Pricing engine of the column-sharded fused loop (spx_fshard_set_lookahead): 0 no look-ahead, 1 look-ahead with
    one pricing kernel per pass, 2 look-ahead with the persistent pricing engine.  `lookahead`: False / True (= by
    world size, unless $SPX_PRICE_ENGINE = `forced` names one) / "per-pass" / "persistent"."""
    if lookahead == "persistent":
        return 2
    if lookahead == "per-pass":
        return 1
    if not lookahead:
        return 0
    if forced in ("per-pass", "persistent"):
        return 2 if forced == "persistent" else 1
    return 2 if 0 < persistent_from <= world else 1


class FusedShardedTableau(ShardedTableau):
    """The column-sharded FUSED loop (csrc/spx_fused.cu, spx_fshard_*): passes of `depth` pivots —
    a whole-GPU cooperative kernel per rank prices them by lazy replay, exchanging keys and the
    winning pivot column from inside the kernel over NVLink peer memory, then every rank streams its
    own columns ONCE for all of them.  Same pivots and bits as every other loop."""

    # World size from which look-ahead uses the persistent pricing engine by default; 0 = never.  Measured on cfg4
    # (profiles/r2/r2q_r2r_persistent_engine.md): 2 ranks 6.4 k pivots/s against 7.0 k with one pricing kernel per pass
    # (the engine keeps 33 SMs for good; the per-pass kernel gives them back to the update between passes), 8 ranks
    # 19.5 k against 19.2-19.3 k (the pricing chain of a level, not the launches around it, bounds the pass) — not a
    # win anywhere, so it stays opt-in.
    PERSISTENT_FROM_WORLD = 0

    def __init__(self, n: int, m: int, rank: int, world: int, device, trace_capacity: int = 0,
                 group=None, rule: int = N.RULE_REFERENCE, depth: int = 8, lookahead=True):
        """lookahead: False — price, update, price, ...; True — the pricing of pass q+1 overlaps the update of
        pass q, as one pricing kernel per pass (and, if PERSISTENT_FROM_WORLD is set, as the persistent pricing engine
        from that many ranks on); "per-pass" / "persistent" force one of the two (every rank must choose the same)."""
        super().__init__(n, m, rank, world, device, trace_capacity=trace_capacity, group=group, rule=rule,
                         lookahead=False)
        L = N.lib()
        self.depth = int(depth)
        self.price_engine = choose_price_engine(lookahead, world, os.environ.get("SPX_PRICE_ENGINE", ""),
                                                self.PERSISTENT_FROM_WORLD)
        self.price_ahead = self.price_engine != 0
        dev = self.device
        wbytes = int(L.spx_fused_workspace_bytes(self.n, max(self.m_loc, 1)))
        self.work = torch.zeros(wbytes // 8 + 16, dtype=torch.float64, device=dev)
        self.xbox = PeerRegion(int(L.spx_fshard_xbox_bytes(self.n, world)), rank, world, dev, group=group)
        self.handle = ctypes.c_void_p()
        with torch.cuda.device(dev):
            N.call("spx_fshard_open", ctypes.byref(self.handle), rank, world, self.n, self.m_loc, self.ld, self.col0,
                   rule, self.A[0].data_ptr(), self.A[1].data_ptr(), self.b[0].data_ptr(), self.b[1].data_ptr(),
                   self.state.data_ptr(), self.work.data_ptr(), self.work.numel() * 8, self.rowlab.data_ptr(),
                   self.collab.data_ptr(), N.ptr(self.trace), self.xbox.ptrs)
            N.call("spx_fshard_set_lookahead", self.handle, self.price_engine)
        self._cur = 0

    def load(self, rows, function, max_pivots: int):
        super().load(rows, function, max_pivots)       # init_state leaves reserved[0] = 0: table 0 in buffer 0
        self._cur = 0

    def load_local(self, block, function_block, max_pivots: int):
        super().load_local(block, function_block, max_pivots)
        self._cur = 0

    def step(self):
        self.run(1)

    def run(self, pivots: int, check_every: int = 0):
        done = 0
        while done < pivots:
            k = pivots - done if check_every <= 0 else min(check_every, pivots - done)
            with torch.cuda.device(self.device):
                N.call("spx_fshard_enqueue", self.handle, k, self.depth,
                       torch.cuda.current_stream(self.device).cuda_stream)
            done += k
            if check_every > 0:
                st = self.read_state()
                if st.status != N.PIVOT:
                    return st
        return None

    def read_state(self) -> N.SpxState:
        st = N.SpxState()
        cur = ctypes.c_int32(0)
        with torch.cuda.device(self.device):
            N.call("spx_fshard_read", self.handle, ctypes.byref(st), ctypes.byref(cur),
                   torch.cuda.current_stream(self.device).cuda_stream)
        self._cur = int(cur.value)
        return st

    def sync(self) -> N.SpxState:
        return self.read_state()

    def solve(self, max_pivots: int, check_every: int = 64):
        while True:
            st = self.run(check_every, check_every=check_every)
            if st is None:
                st = self.read_state()
            if st.status == N.PIVOT and st.npiv >= st.max_pivots:
                self.run(1)                      # the pricing of one more pass reports SPX_CAP or the real ending
                st = self.read_state()
            if st.status != N.PIVOT or st.npiv >= max_pivots:
                return int(st.status), int(st.npiv)

    def local_body(self) -> torch.Tensor:
        self.read_state()
        return self.A[self._cur, :, : self.m_loc]

    def b_current(self) -> torch.Tensor:
        self.read_state()
        return self.b[self._cur, : self.n]

    def pricing_stamps(self) -> np.ndarray:
        """[9, 6] uint64 ns: the phase stamps of the last pricing kernel on this rank (spx_fused_debug_stamps)."""
        out = (ctypes.c_uint64 * 54)()
        with torch.cuda.device(self.device):
            N.call("spx_fused_debug_stamps", self.work.data_ptr(), self.n, self.ld, out, 54,
                   torch.cuda.current_stream(self.device).cuda_stream)
        return np.frombuffer(out, dtype=np.uint64).reshape(9, 6).copy()

    def close(self):
        if self.handle:
            N.call("spx_fshard_close", self.handle)
            self.handle = ctypes.c_void_p()
        self.xbox.close()


class PeerShardedTableau(ShardedTableau):
    """The sharded look-ahead loop enqueued from C (spx_shard_* handle, csrc/spx_shard.cu): per pivot
    no Python, no collective library — update k on the main stream, next b / candidate / NVLink peer
    push / select for pivot k+1 on the handle's side stream."""

    def __init__(self, n: int, m: int, rank: int, world: int, device, trace_capacity: int = 0,
                 group=None, rule: int = N.RULE_REFERENCE):
        super().__init__(n, m, rank, world, device, trace_capacity=trace_capacity, group=group, rule=rule,
                         lookahead=False)
        L = N.lib()
        dev = self.device
        self.lookahead = True
        # the handle wants spx_state[2] and colbuf[2] contiguous
        self.state2 = torch.zeros(2 * ctypes.sizeof(N.SpxState) // 8, dtype=torch.int64, device=dev)
        half = self.state2.numel() // 2
        self.states = [self.state2[:half], self.state2[half:]]
        self.state = self.states[0]
        cb = int(L.spx_colbuf_doubles(self.n))
        self.colbuf2 = torch.zeros(2 * cb, dtype=torch.float64, device=dev)
        self.colbufs = [self.colbuf2[:cb], self.colbuf2[cb:]]
        self.colbuf = self.colbufs[0]
        self.mailboxes = PeerMailboxes(self.n, rank, world, dev, group=group)
        self.handle = ctypes.c_void_p()
        with torch.cuda.device(dev):
            N.call("spx_shard_open", ctypes.byref(self.handle), rank, world, self.n, self.m_loc, self.ld, self.col0,
                   rule, self.A[0].data_ptr(), self.A[1].data_ptr(), self.b[0].data_ptr(), self.b[1].data_ptr(),
                   self.state2.data_ptr(), self.colbuf2.data_ptr(), self.rowlab.data_ptr(), self.collab.data_ptr(),
                   N.ptr(self.trace), self.send.data_ptr(), self.mailboxes.ptrs)
        self._cur = 0

    def load(self, rows, function, max_pivots: int):
        super().load(rows, function, max_pivots)
        N.call("spx_shard_reset", self.handle)
        self._cur = 0

    def load_local(self, block, function_block, max_pivots: int):
        super().load_local(block, function_block, max_pivots)
        N.call("spx_shard_reset", self.handle)
        self._cur = 0

    def step(self):
        self.run(1)

    def run(self, pivots: int, check_every: int = 0):
        done = 0
        while done < pivots:
            k = pivots - done if check_every <= 0 else min(check_every, pivots - done)
            with torch.cuda.device(self.device):
                N.call("spx_shard_enqueue", self.handle, k, torch.cuda.current_stream(self.device).cuda_stream)
            done += k
            if check_every > 0:
                st = self.read_state()
                if st.status != N.PIVOT:
                    return st
        return None

    def read_state(self) -> N.SpxState:
        st = N.SpxState()
        cur = ctypes.c_int32(0)
        with torch.cuda.device(self.device):
            N.call("spx_shard_read", self.handle, ctypes.byref(st), ctypes.byref(cur),
                   torch.cuda.current_stream(self.device).cuda_stream)
        self._cur = int(cur.value)
        self.npiv_enqueued = int(st.npiv) if st.status != N.PIVOT else self.npiv_enqueued
        return st

    def sync(self) -> N.SpxState:
        st = self.read_state()
        self.npiv_enqueued = int(st.npiv)
        return st

    def solve(self, max_pivots: int, check_every: int = 64):
        while True:
            st = self.run(check_every, check_every=check_every)
            if st is None:
                st = self.read_state()
            if st.status != N.PIVOT or st.npiv >= max_pivots:
                return int(st.status), int(st.npiv)

    def close(self):
        if self.handle:
            N.call("spx_shard_close", self.handle)
            self.handle = ctypes.c_void_p()
        self.mailboxes.close(group=self.group)


def solve_batched_sharded(tables: np.ndarray, n: int, m: int, max_pivots: int = 64, rule: str = "reference",
                          rank: Optional[int] = None, world: Optional[int] = None, device=None,
                          solver=None, engine: str = "auto"):
    """Each rank solves its contiguous share of the batch; no collective on the data path.

    Returns (start, count, BatchResult) for this rank.  `solver` defaults to the CUDA
    ``solve_batched``; tests pass a stand-in.  `engine` is passed on to ``solve_batched``
    (and to a stand-in only when it is not "auto").
    """
    if rank is None:
        rank = dist.get_rank() if dist.is_initialized() else 0
    if world is None:
        world = dist.get_world_size() if dist.is_initialized() else 1
    start, count = shard_range(tables.shape[0], rank, world)
    if solver is None:
        from .batched import solve_batched as solver
    kw = {} if engine == "auto" else {"engine": engine}
    res = solver(tables[start:start + count], n, m, max_pivots=max_pivots, rule=rule, device=device, **kw)
    return start, count, res


def cells_range(cells, rank: int, world: int):
    """Contiguous split of LPs with `cells` [B] cells each, balanced by cells: (start, count) of `rank`.

    Rank r starts at the first LP whose prefix sum of cells reaches r/world of the total, so every
    rank holds at most total/world + (the largest LP's cells) cells.
    """
    cells = np.asarray(cells, dtype=np.int64).reshape(-1)
    prefix = np.concatenate([[0], np.cumsum(cells)])
    total = int(prefix[-1])
    bound = lambda r: int(np.searchsorted(prefix * world, r * total, side="left")) if r < world else cells.shape[0]  # noqa: E731
    start = min(bound(rank), cells.shape[0])
    return start, max(0, bound(rank + 1) - start)


def solve_ragged_sharded(lps, max_pivots=64, rule: str = "reference", rank: Optional[int] = None,
                         world: Optional[int] = None, device=None, solver=None, engine: str = "auto",
                         trace: bool = True, snapshots: bool = False):
    """Each rank solves its contiguous, cell-balanced share of a ragged batch; no collective on the data path.

    `lps`, `max_pivots` and `engine` (including "global" and "auto_global") as ``batched.solve_ragged``.
    Returns (start, count, RaggedResult) for this rank.  `solver` defaults to the CUDA ``solve_ragged``;
    tests pass a stand-in.
    """
    from .engine import as_rows_function
    if rank is None:
        rank = dist.get_rank() if dist.is_initialized() else 0
    if world is None:
        world = dist.get_world_size() if dist.is_initialized() else 1
    lps = [as_rows_function(cons, fn) for cons, fn in lps]
    start, count = cells_range([r.size + c.size for r, c in lps], rank, world)
    caps = np.asarray(max_pivots, dtype=np.int64)
    caps = int(caps) if caps.ndim == 0 else caps[start:start + count]
    if solver is None:
        from .batched import solve_ragged as solver
    res = solver(lps[start:start + count], max_pivots=caps, rule=rule, trace=trace, snapshots=snapshots,
                 device=device, engine=engine)
    return start, count, res
