#!/usr/bin/env python
"""bench.py — pivots/sec + tableau-update HBM GB/s on the BASELINE.json workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload): cfg4 of BASELINE.json — the dense 16384 x 32768 fp64 LP
D(16384, 32768, seed 0) of SURVEY.md §8d.  One *step* = PIVOTS_PER_STEP (1000) consecutive
pivots of that tableau.  The full solve needs ~1e6 pivots, so timed steps simply continue the same
solve.  EVERY timed pivot is checked: the pivot sequence of the whole run, and the b column, f row and a
64-bit checksum of the 4.3 GB body after the last timed pivot, against oracle marks generated offline
(tests/golden/cfg4_long.json, made by tests/golden/make_cfg4_long.py) before anything is printed.

  value   pivots/s with the tableau resident in HBM (CUDA events, max over ranks); the loop is the fused
          one: 8 pivots priced from the stored table, then ONE stream over the body applies them all
  e2e     pivots/s through the public API (SimplexMethod(rows, c).solve(...)) with the
          4.3 GB tableau in PINNED HOST memory: upload + pivots + result read-back
  roofline  the dominant kernel (update_lazy_kernel): 16 B x cells per LAUNCH / its CUDA-event duration, plus
          its fp64-issue fraction (the binding roofline at 8 pivots per pass);
          roofline_single_pivot_kernel: the one-pivot-per-pass streaming kernel (16 B per cell per pivot —
          the north star's roofline)
  cpu_baseline  oracle/spx_oracle.c (a C port of the reference's loop, OpenMP on all host cores) on this host;
          cpu_baseline_reference: the reference's own simplex.py where $SIMPLEX_REF points at its sources
          (pure Python, it cannot travel to the GPU box)
  legs    the other BASELINE configs that fit one line: cfg1 (GUI LP through get_solution()), cfg2 (1000 x 2000,
          L2-resident), cfg3 (65,536 small LPs, plus a 1,048,576-LP batch), cfg5 (Klee-Minty n = 20)

N > 1 (torchrun): the body is column-sharded, one process per GPU; per pivot the ranks exchange their entering
keys and candidate columns over NVLink peer memory from inside the pricing kernel (strong scaling: the tableau is
fixed); before timing, every rank runs a committed "late" LP whose entering column changes owner rank > 100 times
and compares trace, b, f and body with the oracle's golden; the cfg3 batch is split over the ranks, no collective.
--impl reference: the reference's algorithm on the host cores (the oracle port with all host threads; the
reference itself is pure Python and cannot travel to the GPU box), same config, a bounded sample of each step.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_ROWS, M_COLS, SEED = 16384, 32768, 0
PIVOTS_PER_STEP = 1000
DUMP_SAMPLE_CELLS = 1 << 20        # body cells --dump-outputs samples (the cfg4 body is 4.3 GB)
METRIC = "pivots/sec (16k x 32k fp64 tableau)"
UNIT = "pivots/s"
GOLDEN = os.path.join(ROOT, "tests", "golden")


def cells(n, m):
    return n * (m + 1) + m


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy_ burst)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def golden_cfg4():
    """(input sha256, trace [K][2] int32, marks {pivot count: {pivot_sha256, b_sha256, f_sha256, body_checksum_u64}})
    — the long oracle prefix when it is there, else the 2000-pivot prefix of cfg_digests.json."""
    with open(os.path.join(GOLDEN, "cfg_digests.json")) as fh:
        g = json.load(fh)["cfg4"]
    trace, marks = np.asarray(g["trace"], dtype=np.int32), dict(g["marks"])
    lp, tp = os.path.join(GOLDEN, "cfg4_long.json"), os.path.join(GOLDEN, "cfg4_long_trace.npy")
    if os.path.exists(lp) and os.path.exists(tp):
        with open(lp) as fh:
            gl = json.load(fh)
        tl = np.load(tp)
        assert gl["input_sha256"] == g["input_sha256"] and (tl[: len(trace)] == trace).all()
        trace, marks = tl, gl["marks"]
    return g["input_sha256"], trace, {int(k): v for k, v in marks.items()}


def as_i64(v: int) -> int:
    """An unsigned 64-bit checksum as the int64 a torch tensor holds (same bits; sums wrap the same way)."""
    v &= 0xFFFFFFFFFFFFFFFF
    return v - (1 << 64) if v >= (1 << 63) else v


def check_against_marks(trace_np, need, marks, gold, table_at_need=None):
    """Assert the run's pivot sequence against the golden trace (all `need` pivots when the golden is that long) and,
    when `need` is a mark, the table digests.  Returns the parity string of the JSON line."""
    from simplex_method_solver_b200 import workloads as W
    k = min(need, len(gold))
    assert (trace_np[:k] == gold[:k]).all(), "pivot sequence differs from the golden prefix"
    what = [f"pivot sequence == oracle golden for the first {k} of {need} pivots of the run"]
    mk = marks.get(need)
    if mk is not None and k == need:
        assert W.pivot_digest(trace_np[:need]) == mk["pivot_sha256"]
        what = [f"pivot sequence == oracle golden for ALL {need} pivots of the run (sha256 mark at pivot {need})"]
        if table_at_need is not None and "body_checksum_u64" in mk:
            b_sha, f_sha, body_ck = table_at_need()
            assert b_sha == mk["b_sha256"], "b column after the last timed pivot differs from the oracle mark"
            assert f_sha == mk["f_sha256"], "f row after the last timed pivot differs from the oracle mark"
            assert body_ck == int(mk["body_checksum_u64"]), "body checksum after the last timed pivot differs"
            what.append(f"b column sha256, f row sha256 and the 64-bit checksum of all {N_ROWS * M_COLS} body cells "
                        f"after pivot {need} == oracle marks (tests/golden/cfg4_long.json)")
    return "; ".join(what)


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU while the timed region runs (NVML)."""

    def __init__(self, index: int, period: float = 0.1):
        self.index, self.period = index, period
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = int(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {
                getattr(nv, "nvmlClocksEventReasonGpuIdle", 0x1): "gpu_idle",
                getattr(nv, "nvmlClocksEventReasonApplicationsClocksSetting", 0x2): "applications_clocks_setting",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonSyncBoost", 0x10): "sync_boost",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
            }
            while not self._stop.is_set():
                self.sm.append(int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                for bit, name in names.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
                self._stop.wait(self.period)
        except Exception as e:  # NVML missing: report that instead of inventing numbers
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def __enter__(self):
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thr.join(timeout=2)

    def summary(self):
        return {"sm_mhz": int(statistics.median(self.sm)) if self.sm else None,
                "sm_max_mhz": self.max_mhz, "samples": len(self.sm), "reasons": sorted(self.reasons)}


def config_dict():
    """The WORKLOAD, identical for both arms and every N; how each arm runs it is under "implementation"."""
    return {"workload": "cfg4: dense LP D(n=16384, m=32768, seed=0), fp64 tableau 4.295 GB (x2 ping-pong)",
            "n": N_ROWS, "m": M_COLS, "cells": cells(N_ROWS, M_COLS),
            "pivots_per_step": PIVOTS_PER_STEP,
            "step": "1000 consecutive pivots of the same solve (the reference arm times a bounded sample of each step)",
            "l2_policy": "inputs (8.6 GB per pivot / per pass) far exceed the 126 MB L2; no flush needed",
            "rule": "reference (first-negative entering, max-negative-ratio leaving)"}


def implementation_dict(ngpu, exchange="fused", fallback=None, price_engine=None):
    d = {"loop": "fused: 8 pivots priced from the stored table (coop_price_kernel), then ONE stream over the body applies "
                 "them (update_lazy_kernel, csrc/spx_fused.cu)" if ngpu == 1 else
                 "fused, column-sharded: cooperative pricing with the in-kernel NVLink exchange of keys and the pivot "
                 "column (shard_price_kernel), then one stream over the local columns per 8 pivots" if exchange == "fused" else
                 "pivot at a time, column-sharded: look-ahead pricing of pivot k+1 during update k (csrc/spx_shard.cu, spx_pick.cu)",
         "parallelism": "single GPU" if ngpu == 1 else
         f"column-sharded x{ngpu}, one key + candidate-column exchange per pivot over NVLink peer memory"}
    if ngpu > 1:
        d["exchange"] = exchange
    if fallback:
        d["exchange_fallback"] = fallback
    if os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS"):
        d["cuda_device_max_connections"] = os.environ["CUDA_DEVICE_MAX_CONNECTIONS"]
    if price_engine:
        d["price_engine"] = price_engine + (
            ": ONE cooperative pricing kernel per run() call stays resident and hands passes to the update kernels "
            "through device flags" if price_engine == "persistent" else
            ": one cooperative pricing kernel per pass on a high-priority side stream, events between it and the "
            "update kernels" if price_engine == "per-pass" else "")
    return d


# ------------------------------------------------------------------------------ reference arm
def host_threads() -> int:
    """All the host threads this process may use — NOT $OMP_NUM_THREADS (torchrun exports OMP_NUM_THREADS=1)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def python_reference_timings(budget_s=2.0):
    """The reference's OWN simplex.py on this host (1 core: pure Python), where its sources are reachable through
    $SIMPLEX_REF (the build container; the GPU box has no copy and sources are never vendored into this repo).
    Loop timed: pick_element() + recalculate_matrix() (the pattern of simplex.py:261-269)."""
    src = os.environ.get("SIMPLEX_REF", "")
    path = os.path.join(src, "simplex.py") if src else ""
    if not path or not os.path.exists(path):
        return {"unavailable": "the reference is pure Python and does not travel to the GPU box; set $SIMPLEX_REF to its "
                               "src/ directory to time it (done in the build container: profiles/r2/python_reference_build_container.json)"}
    import importlib.util
    from simplex_method_solver_b200 import workloads as W
    spec = importlib.util.spec_from_file_location("reference_simplex", path)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)

    def drive(rows, c, max_s=None, max_piv=None):
        sm = ref.SimplexMethod([list(map(float, r)) for r in rows], [float(v) for v in c])
        k, t0 = 0, time.perf_counter()
        while True:
            ok, *_ = sm.pick_element()
            if not ok:
                break
            sm.recalculate_matrix()
            k += 1
            if (max_piv and k >= max_piv) or (max_s and time.perf_counter() - t0 > max_s):
                break
        return k, time.perf_counter() - t0

    out = {"kind": "reference", "cores": 1, "host_cores": host_threads(),
           "loop": "pick_element() + recalculate_matrix() of the reference's simplex.py (pattern of simplex.py:261-269)"}
    reps = 200
    t0 = time.perf_counter()
    for _ in range(reps):
        k1, _ = drive(W.CFG1_ROWS, W.CFG1_C)
    dt = (time.perf_counter() - t0) / reps
    out["cfg1"] = {"pivots": k1, "solves_per_s": 1.0 / dt, "pivots_per_s": k1 / dt, "sample": f"{reps} full solves"}
    t0 = time.perf_counter()
    for _ in range(reps):
        ref.SimplexMethod([list(map(float, r)) for r in W.CFG1_ROWS], [float(v) for v in W.CFG1_C]).get_solution()
    out["cfg1"]["get_solution_per_s"] = reps / (time.perf_counter() - t0)     # what the GUI calls (snapshots included)
    T, C = W.gui_batch(4096, 0)
    t0 = time.perf_counter()
    piv = sum(drive(T[k], C[k])[0] for k in range(4096))
    dt = time.perf_counter() - t0
    out["cfg3"] = {"lps_per_s": 4096 / dt, "pivots_per_s": piv / dt, "sample": "first 4,096 of the 65,536 LPs"}
    rows, c = W.klee_minty(20)
    k5, dt = drive(rows, c, max_s=budget_s)
    out["cfg5"] = {"pivots_per_s": k5 / dt, "sample": f"first {k5} pivots ({budget_s:.0f} s) of the 1,048,575"}
    rows, c = W.dense_lp(1000, 2000, 0)
    k2, dt = drive(rows, c, max_piv=1)
    out["cfg2"] = {"pivots_per_s": k2 / dt, "sample": "first pivot of the 13,579",
                   "cells_per_s": cells(1000, 2000) * k2 / dt}
    out["cfg4"] = {"pivots_per_s_extrapolated": out["cfg2"]["cells_per_s"] / cells(N_ROWS, M_COLS),
                   "sample": "NOT runnable as nested lists (~40 GB); extrapolated from the cfg2 cells/s"}
    return out


def run_reference(args):
    """The reference's algorithm on the host cores: oracle/spx_oracle.c (C port, OpenMP on all host threads)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from simplex_method_solver_b200 import workloads as W
    oracle.build()
    threads = host_threads()
    oracle.lib().orc_set_num_threads(threads)          # torchrun exports OMP_NUM_THREADS=1: do not inherit it
    if args.python_reference_only:
        print(json.dumps({"impl": "reference", "cpu_baseline_reference": python_reference_timings()}), flush=True)
        return
    per_step = max(1, args.ref_pivots_per_step)
    log(f"[reference] generating D({N_ROWS},{M_COLS},{SEED}) ... ({threads} threads)")
    rows, c = W.dense_lp(N_ROWS, M_COLS, SEED)
    T = np.concatenate([rows.reshape(-1), c])
    del rows
    Nn = np.empty_like(T)
    L = oracle.lib()
    _, gold, _ = golden_cfg4()
    k = 0

    def step():
        nonlocal T, Nn, k
        for _ in range(per_step):
            st, r, cc, _e = oracle.pick(T, N_ROWS, M_COLS)
            assert st == oracle.PIVOT
            if k < len(gold):
                assert (r, cc) == tuple(gold[k]), "oracle diverged from its own golden trace"
            L.orc_update(oracle._dp(T), oracle._dp(Nn), N_ROWS, M_COLS, r, cc)
            T, Nn = Nn, T
            k += 1

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = (f"{per_step} of each step's {PIVOTS_PER_STEP} pivots x {args.steps} steps of the same 16384x32768 tableau "
              f"(oracle/spx_oracle.c, OpenMP {threads} threads set explicitly; the reference itself is "
              f"single-threaded pure Python, ~1.5e6 cells/s)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_dict(),
        "implementation": {"loop": "pick_element() then recalculate_matrix(), one pivot at a time, out of place "
                                   "(oracle/spx_oracle.c: orc_pick + orc_update)",
                           "parallelism": f"OpenMP over tableau rows, {threads} host threads",
                           "pivots_timed_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "cpu_baseline_reference": python_reference_timings(),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ our arm
def cpu_baseline_sample(rows, c, gold, budget_s=20.0):
    """oracle port timed on a bounded sample of the same workload (rank 0, N=1 only)."""
    import oracle
    oracle.build()
    threads = host_threads()
    oracle.lib().orc_set_num_threads(threads)
    T = np.concatenate([rows.reshape(-1), c])
    Nn = np.empty_like(T)
    L = oracle.lib()
    done, t_used = 0, 0.0
    # one untimed pivot to fault the pages in
    while True:
        t0 = time.perf_counter()
        st, r, cc, _e = oracle.pick(T, N_ROWS, M_COLS)
        assert st == oracle.PIVOT and (r, cc) == tuple(gold[done])
        L.orc_update(oracle._dp(T), oracle._dp(Nn), N_ROWS, M_COLS, r, cc)
        T, Nn = Nn, T
        dt = time.perf_counter() - t0
        done += 1
        if done > 1:
            t_used += dt
        if t_used > budget_s or done >= 64:
            break
    timed = done - 1
    return {"value": timed / t_used, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"first {timed} pivots (after 1 untimed) of the same 16384x32768 tableau, "
                      f"oracle/spx_oracle.c with OpenMP on {threads} threads"}


def dump_outputs(out_dir, tab, status, npiv, last_step):
    """--dump-outputs: what a caller of the timed loop holds after its last step, one float64 .npy per array: the
    step's pivots, the b column, the f row, x / objective / labels (DeviceTableau.solution()) and a fixed seeded sample
    of the body cells with their row-major indices.  The inputs are seeded, so two builds run with the same arguments
    can be compared file for file."""
    import torch
    n, m = tab.n, tab.m
    cur = tab.cur(npiv)
    sol = tab.solution(status, npiv)
    index = np.unique(np.random.default_rng(SEED).integers(0, n * m, DUMP_SAMPLE_CELLS))
    r, c = np.divmod(index, m)
    sample = tab.A[cur].view(-1)[torch.from_numpy(r * tab.ld + c).to(tab.device)]
    arrays = {"status": [status, npiv], "trace": sol.trace[max(0, npiv - last_step): npiv],
              "b": tab.b[cur, :n], "f_row": tab.A[cur, n, :m], "x": sol.x, "objective": [sol.obj2, sol.objective],
              "row_labels": sol.rowlab, "column_labels": sol.collab, "body_sample_index": index, "body_sample": sample}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))
    return sorted(arrays)


def batched_leg(dev, rank, world, dist=None, reps=20, B=65536, golden=True):
    """cfg3 of BASELINE.json: B independent 2-var / 8-constraint LPs, one warp per LP, the batch
    split contiguously over the ranks with no collective (unit: LPs; total work fixed).
    The kernel is timed DIRECTLY: `reps` device copies of this rank's share (rotated, so each launch reads tables
    that are not in L2), restores outside the events.  Returns the dict reported under "batched" (rank 0)."""
    import torch
    from simplex_method_solver_b200 import workloads as W
    from simplex_method_solver_b200.batched import DeviceBatch
    from simplex_method_solver_b200.parallel import shard_range
    n, m = 8, 2
    T, C = W.gui_batch(B, 0)
    tabs = W.batch_flat(T, C)
    start, count = shard_range(B, rank, world)
    pinned = torch.from_numpy(tabs[start:start + count].copy()).pin_memory()
    db = DeviceBatch(count, n, m, max_pivots=64, trace=True, device=dev)
    out_x = torch.empty((count, m), dtype=torch.float64).pin_memory()
    out_st = torch.empty(count, dtype=torch.int32).pin_memory()
    staged = pinned.to(dev)
    nbuf = max(2, min(reps, (512 << 20) // max(staged.numel() * 8, 1)))
    ring = [torch.empty_like(db.T) for _ in range(nbuf)]
    home = db.T

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def max_ranks(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- resident: kernel only
    for buf in ring:
        buf[:count].copy_(staged)
    for i in range(3):                                   # warm-up (also consumes ring[0..2])
        db.T = ring[i % nbuf]
        db.run()
    sync_all()
    ker = []
    done = 0
    while done < reps:
        k = min(nbuf, reps - done)
        for buf in ring[:k]:
            buf[:count].copy_(staged)                    # untimed restore (the solver works in place)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for buf in ring[:k]:
            db.T = buf
            db.run()
        e1.record()
        sync_all()
        ker.append((e0.elapsed_time(e1), k))
        done += k
    ker_ms = max_ranks(sum(t for t, _ in ker) / sum(k for _, k in ker))
    db.T = home
    del ring

    # ---- end to end: pinned upload + kernel + result read-back
    def e2e():
        db.upload(pinned, non_blocking=True)
        db.run()
        out_x.copy_(db.x[:count], non_blocking=True)
        out_st.copy_(db.status[:count], non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(3):
        e2e()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(reps):
        e2e()
    sync_all()
    ms_e2e = max_ranks(1e3 * (time.perf_counter() - t0) / reps)
    res = db.result()
    piv = torch.tensor([int(res.npiv.sum()), int((res.status == 0).sum())], dtype=torch.int64, device=dev)
    if dist is not None:
        dist.all_reduce(piv)
    total_piv, n_opt = int(piv[0].item()), int(piv[1].item())
    parity = f"{total_piv:,} pivots, {n_opt:,} optimal"
    if golden:
        assert total_piv == 408212 and n_opt == B, (total_piv, n_opt)     # golden: tests/golden/cfg_digests.json
        parity = "408,212 pivots, all optimal == golden"
    else:
        assert n_opt == B, (n_opt, B)
    return {"workload": f"cfg3 shape: {B:,} LPs (8 constraints x 2 vars), one warp per LP, split over ranks, no collective",
            "lps_per_s": B / (ker_ms * 1e-3), "pivots_per_s": total_piv / (ker_ms * 1e-3), "kernel_ms": ker_ms,
            "timing": f"kernel alone, CUDA events around {reps} launches on rotating device copies (restores untimed), max over ranks",
            "e2e_lps_per_s": B / (ms_e2e * 1e-3), "e2e_ms": ms_e2e,
            "h2d_bytes": int(pinned.numel() * 8), "d2h_bytes": int(out_x.numel() * 8 + out_st.numel() * 4),
            "northstar_convention_GBps": 16.0 * 26 * total_piv / (ker_ms * 1e-3) / 1e9,
            "parity": parity}


def resident_leg(dev):
    """cfg2 of BASELINE.json: dense 1000 x 2000 LP (16 MB, L2-resident), solved to optimality by the
    persistent cooperative kernel (csrc/spx_resident.cu); full pivot sequence checked against the golden digest."""
    import torch
    from simplex_method_solver_b200 import workloads as W
    from simplex_method_solver_b200.engine import DeviceTableau
    from simplex_method_solver_b200.simplex import SimplexMethod
    with open(os.path.join(GOLDEN, "cfg_digests.json")) as fh:
        g = json.load(fh)["cfg2"]["oracle_full"]
    rows, c = W.dense_lp(1000, 2000, 0)
    best = None
    for it in range(3):
        tab = DeviceTableau(1000, 2000, device=dev, trace_capacity=20000)
        tab.load(rows, c, max_pivots=20000)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st, npiv = tab.solve(lookahead="resident")
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    assert st == 0 and npiv == g["npiv"] == 13579
    assert W.pivot_digest(tab.trace[:npiv].cpu().numpy()) == g["pivot_sha256_final"]
    # end to end through the public API: pinned host rows in, x / objective / trace out
    pinned = torch.from_numpy(rows).pin_memory()
    e2e_t = []
    for it in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sm = SimplexMethod(pinned.numpy(), c, device=dev, engine="stream")
        sol = sm.solve(max_pivots=20000, chunk=20000)
        torch.cuda.synchronize()
        e2e_t.append(time.perf_counter() - t0)
        assert sol.npiv == npiv and sol.status == 0 and float(sol.objective).hex() == g["objm"]
    e2e_s = min(e2e_t[1:])
    cells2 = cells(1000, 2000)
    ceiling = measured_peak()[0] * 1e9 / (16.0 * cells2)
    return {"workload": "cfg2: dense LP D(1000, 2000, seed 0) to optimality, 13,579 pivots, persistent L2-resident kernel",
            "pivots_per_s": npiv / (best * 1e-3), "ms": best, "us_per_pivot": 1e3 * best / npiv,
            "northstar_convention_GBps": 16.0 * cells2 * npiv / (best * 1e-3) / 1e9,
            "frac_of_convention_ceiling": (npiv / (best * 1e-3)) / ceiling,
            "convention_ceiling_pivots_per_s": ceiling,
            "e2e_pivots_per_s": npiv / e2e_s, "e2e_ms": 1e3 * e2e_s,
            "e2e_api": "SimplexMethod(pinned_rows, c).solve(): upload 16 MB + solve + x/objective/trace read-back",
            "parity": "13,579 pivots, sha256 of the pivot sequence == golden; objective bits == golden"}


def small_legs(dev):
    """cfg1 (the reference's own 4 x 2 GUI LP through get_solution(), every Info compared with the reference's
    snapshots) and cfg5 (Klee-Minty n = 20: 1,048,575 sequential pivots in one CTA-resident launch)."""
    import torch
    from simplex_method_solver_b200 import workloads as W
    from simplex_method_solver_b200.batched import DeviceBatch
    from simplex_method_solver_b200.simplex import Error, SimplexMethod
    with open(os.path.join(GOLDEN, "cfg_digests.json")) as fh:
        dig = json.load(fh)
    with open(os.path.join(GOLDEN, "reference_cases.json")) as fh:
        case = next(cc for cc in json.load(fh)["cases"] if cc["name"] == "ref_example_cfg1_205")
    # ---- cfg1
    reps = 50
    infos = SimplexMethod(W.CFG1_ROWS, W.CFG1_C, device=dev).get_solution()      # warm-up + parity
    assert not any(isinstance(i, Error) for i in infos)
    assert [[i.i, i.j] for i in infos[:-1]] == case["trace"]
    assert W.snapshot_digest([i.table for i in infos]) == case["snapshot_sha256"]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        SimplexMethod(W.CFG1_ROWS, W.CFG1_C, device=dev).get_solution()
    dt = (time.perf_counter() - t0) / reps
    cfg1 = {"workload": "cfg1: the reference's own 4-constraint / 2-variable GUI LP (simplex.py:205-209)",
            "solves_per_s": 1.0 / dt, "ms_per_solve": 1e3 * dt, "pivots": len(infos) - 1,
            "api": "SimplexMethod(constraints, function).get_solution(): upload, one warp-resident launch, 5 Info snapshots back",
            "parity": "pivots, labels and sha256 of all 5 snapshot tables == the reference's get_solution()"}
    # ---- cfg5
    g = dig["km20"]
    rows, c = W.klee_minty(20)
    flat = torch.from_numpy(np.concatenate([rows.reshape(-1), c])[None, :]).to(dev)
    db = DeviceBatch(1, 20, 20, max_pivots=1 << 20, trace=True, device=dev)
    best = None
    for it in range(2):
        db.T.copy_(flat)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        db.run()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    npiv = int(db.npiv[0].item())
    assert npiv == g["npiv"] == (1 << 20) - 1 and int(db.status[0].item()) == 0
    assert W.pivot_digest(db.trace[0, :npiv].cpu().numpy()) == g["pivot_sha256"]
    assert hashlib.sha256(db.T[0].cpu().numpy().tobytes()).hexdigest() == g["final_table_sha256"]
    cfg5 = {"workload": "cfg5: Klee-Minty n = 20, 1,048,575 sequential pivots, one CTA-resident launch (batched_kernel<1>)",
            "pivots_per_s": npiv / (best * 1e-3), "ms": best, "us_per_pivot": 1e3 * best / npiv,
            "northstar_convention_GBps": 16.0 * 440 * npiv / (best * 1e-3) / 1e9,
            "parity": "1,048,575 pivots, sha256 of the pivot sequence and of the final table == the reference's"}
    return cfg1, cfg5


def fused_depth_for(world: int) -> int:
    """Pivots per pass of the sharded fused loop: 8 everywhere (measured; see profiles/README.md)."""
    return 8


def late_lp_preflight(FusedCls, rank, world, dev, dist):
    """N > 1 parity proof the driver's 1-GPU test box cannot run: a committed LP whose entering column starts on the
    LAST column block and changes owner rank > 100 times (tests/golden/late_lp.json, oracle-generated), through the
    fused sharded loop on every rank; trace, b, f and every body cell compared with the oracle's golden.
    Returns (ok, owner_changes, why)."""
    import torch
    from simplex_method_solver_b200 import _native as N
    from simplex_method_solver_b200 import workloads as W
    from simplex_method_solver_b200.parallel import column_block
    with open(os.path.join(GOLDEN, "late_lp.json")) as fh:
        g = json.load(fh)
    n, m, cap = g["n"], g["m"], g["npiv"]
    rows, c = W.dense_lp(n, m, g["seed"])
    c[: int(0.95 * m)] = np.abs(c[: int(0.95 * m)])                  # tests/util.py::make_lp(..., "late")
    assert W.input_digest(rows, c) == g["input_sha256"]
    gold = np.asarray(g["trace"], dtype=np.int32)
    blocks = [column_block(m, r, world) for r in range(world)]
    own = [next(k for k, (a, w) in enumerate(blocks) if a <= int(cc) < a + w) for _, cc in gold]
    changes = sum(1 for a, b in zip(own, own[1:]) if a != b)
    # local work first (anything may fail on ONE rank), then the same collectives on EVERY rank whatever happened
    why, sh, ck_local, f_local, b_sha = "", None, 0, b"", ""
    try:
        sh = FusedCls(n, m, rank, world, device=dev, trace_capacity=cap + 64, depth=fused_depth_for(world))
        sh.load(rows, c, max_pivots=cap + 64)
        sh.solve(cap + 64, check_every=64)
        st = sh.sync()
        if (int(st.status), int(st.npiv)) != (g["status"], g["npiv"]):
            why = f"late LP ended with status {st.status} after {st.npiv} pivots, golden {g['status']} after {g['npiv']}"
        elif not (sh.trace[: g["npiv"]].cpu().numpy() == gold).all():
            why = "late LP: pivot sequence differs from the oracle's"
        else:
            body = sh.local_body()
            ck_local = as_i64(W.body_checksum_torch(body[:n], m_total=m, col0=sh.col0)) if sh.m_loc else 0
            f_local = body[n].cpu().numpy().tobytes()
            b_sha = hashlib.sha256(sh.b_current().cpu().numpy().tobytes()).hexdigest()
    except Exception as e:                               # noqa: BLE001 - reported, then the documented fallback
        why = f"{type(e).__name__}: {e}"
    finally:
        if sh is not None:
            try:
                sh.close()
            except Exception:                            # noqa: BLE001
                pass
    ck = torch.tensor([ck_local], dtype=torch.int64, device=dev)
    dist.all_reduce(ck)
    fs = [None] * world
    dist.all_gather_object(fs, f_local)
    if not why:
        if (int(ck.item()) & 0xFFFFFFFFFFFFFFFF) != int(g["body_checksum_u64"]):
            why = "late LP: body checksum differs from the oracle's"
        elif hashlib.sha256(b"".join(fs)).hexdigest() != g["f_sha256"]:
            why = "late LP: f row differs from the oracle's"
        elif b_sha != g["b_sha256"]:
            why = "late LP: b column differs from the oracle's"
    okf = torch.tensor([0 if why else 1], dtype=torch.int32, device=dev)
    dist.all_reduce(okf, op=dist.ReduceOp.MIN)
    return int(okf.item()) == 1, changes, why


def run_ours(args):
    import torch
    import torch.distributed as dist
    from simplex_method_solver_b200 import _native as N
    from simplex_method_solver_b200 import workloads as W
    from simplex_method_solver_b200.engine import DeviceTableau
    from simplex_method_solver_b200.simplex import SimplexMethod

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        # a rank that fails an assertion must not leave its peers in a collective for NCCL's default 10 minutes
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    N.lib()
    if args.shard_threads:
        assert N.load().spx_set_option(13, args.shard_threads) == 0
    if args.shard_ctas:
        assert N.load().spx_set_option(14, args.shard_ctas) == 0
    peak, peak_src = measured_peak()
    in_sha, gold, marks = golden_cfg4()

    log(f"[rank {rank}] generating D({N_ROWS},{M_COLS},{SEED}) ...")
    t0 = time.perf_counter()
    rows, c = W.dense_lp(N_ROWS, M_COLS, SEED)
    log(f"[rank {rank}] generated in {time.perf_counter() - t0:.1f}s")
    P = PIVOTS_PER_STEP
    need = (args.warmup + args.steps) * P

    if world == 1:
        # ---------------- value: tableau resident in HBM --------------------------------
        tab = DeviceTableau(N_ROWS, M_COLS, device=dev, trace_capacity=need + 64)
        tab.load(rows, c, max_pivots=need + 64)   # the cap is never reached inside the timed region
        for _ in range(args.warmup):
            st, npiv = tab.solve(chunk=P, stop_after=P)
        torch.cuda.synchronize()
        N.load().spx_launch_count(1)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local) as clk:
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(args.steps):
                st, npiv = tab.solve(chunk=P, stop_after=P)
            ev1.record()
            torch.cuda.synchronize()
        launches = int(N.load().spx_launch_count(0))
        total_ms = ev0.elapsed_time(ev1)
        if args.dump_outputs:                             # before the checks, so a diverging build is dumped too
            names = dump_outputs(args.dump_outputs, tab, st, npiv, P)
            log(f"[rank {rank}] wrote {', '.join(names)} (.npy) to {args.dump_outputs}")
        assert npiv == need and st == N.PIVOT, (st, npiv)
        tr = tab.trace[:need].cpu().numpy()

        def table_digests():
            cur = need & 1                                # spx_solve leaves table k in buffer k & 1
            b_sha = hashlib.sha256(tab.b[cur, :N_ROWS].cpu().numpy().tobytes()).hexdigest()
            f_sha = hashlib.sha256(tab.A[cur, N_ROWS, :M_COLS].cpu().numpy().tobytes()).hexdigest()
            return b_sha, f_sha, W.body_checksum_torch(tab.A[cur, :N_ROWS, :M_COLS])

        parity = check_against_marks(tr, need, marks, gold, table_digests)
        value = args.steps * P / (total_ms * 1e-3)

        # ---------------- roofline 1: the dominant kernel of the timed loop = the fused update (K6):
        # one launch streams the body once (16 B per cell) and applies FUSE_DEPTH pivots to every cell
        # timed INSIDE a long back-to-back run (150 passes, ~0.3 s; the mean is over the last 100): the loop is power
        # capped (sw_power_cap, ~1 kW), and a short burst would be measured at clocks the timed steps never see
        nmeas, nskip = 150, 50
        F = int(N.load().spx_get_option(N.OPT_FUSE_DEPTH)) or 8
        st_obj = tab.read_state()
        st_obj.max_pivots = need + (nmeas + 3) * F + 64
        st_obj.reserved[0] = need & 1
        tab.write_state(st_obj)
        tab.trace = None
        fe = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(nmeas)]
        with ClockSampler(local) as clk_k:
            for q in range(nmeas):
                fe[q][0].record()
                tab.fused_pass(F, 1)                         # the pricing kernel (whole-GPU cooperative)
                fe[q][1].record()
                tab.fused_pass(F, 2)                         # the fused streaming update
                fe[q][2].record()
            torch.cuda.synchronize()
        price_ms = statistics.mean(e[0].elapsed_time(e[1]) for e in fe[nskip:])
        fused_ms = statistics.mean(e[1].elapsed_time(e[2]) for e in fe[nskip:])
        st_obj = tab.read_state()
        assert st_obj.status == N.PIVOT and st_obj.npiv == need + nmeas * F, (st_obj.status, st_obj.npiv)
        fused_npiv, fused_cur = int(st_obj.npiv), int(st_obj.reserved[0]) & 1
        alg_bytes = 16.0 * cells(N_ROWS, M_COLS)
        achieved = alg_bytes / (fused_ms * 1e-3) / 1e9
        sm_mhz = clk_k.summary()["sm_mhz"] or clk.summary()["sm_mhz"] or 0     # the clock DURING these launches
        dp_ops = 6.0 * cells(N_ROWS, M_COLS) * F          # 2 DMUL + DADD + DMUL + 2 DFMA per cell per pivot
        dp_peak = 148 * 64 * sm_mhz * 1e6                 # fp64 issue slots/s at the SM clock seen under load
        traffic = None
        tp = os.path.join(ROOT, "profiles", "update_kernel_traffic.json")
        if os.path.exists(tp):
            with open(tp) as fh:
                traffic = json.load(fh).get("fused_dram_bytes_per_launch")
        step_ms = total_ms / args.steps
        roofline = {"bound": "hbm", "kernel": f"update_lazy_kernel (K6: {F} pivots per pass over the body)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "peak_source": peak_src, "traffic": traffic,
                    "algorithmic_bytes_per_launch": alg_bytes, "pivots_per_launch": F,
                    "kernel_ms": fused_ms, "pricing_kernel_ms": price_ms,
                    "kernel_timing": f"CUDA events around each of the last {nmeas - nskip} of {nmeas} back-to-back passes (sustained, power capped)",
                    "clocks_during_kernel_timing": clk_k.summary(),
                    "kernel_share_of_step": fused_ms * (P / F) / step_ms,
                    "northstar_convention_GBps": alg_bytes * F / (fused_ms * 1e-3) / 1e9,
                    "fp64_pipe": {"achieved_Gops": dp_ops / (fused_ms * 1e-3) / 1e9,
                                  "peak_Gops_at_measured_clock": dp_peak / 1e9,
                                  "frac": (dp_ops / (fused_ms * 1e-3)) / dp_peak if dp_peak else None,
                                  "sm_mhz": sm_mhz,
                                  "fp64_issues_per_cell_per_pivot": 6},
                    "note": "F dependent rank-1 updates per cell in registers: HBM moves 16 B per cell per PASS, so at F=8 "
                            "the kernel is fp64-issue bound (fp64_pipe.frac is the binding roofline), not HBM bound; the "
                            "single-pivot streaming kernel is below"}

        # ---------------- roofline 2: the single-pivot streaming kernel K3 (the 16 B/cell/pivot roofline)
        st_obj.max_pivots = fused_npiv + 64
        st_obj.reserved[0] = 0
        tab.write_state(st_obj)
        if fused_cur != (fused_npiv & 1):                 # restore "table k lives in buffer k & 1"
            tab.A[fused_npiv & 1].copy_(tab.A[fused_cur])
            tab.b[fused_npiv & 1].copy_(tab.b[fused_cur])
        nk3 = 40
        tab2_npiv = fused_npiv
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nk3)]
        pick_evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nk3)]
        for q in range(nk3):
            pick_evs[q][0].record()
            tab.pick(tab2_npiv, sticky=True)
            pick_evs[q][1].record()
            evs[q][0].record()
            tab.update(tab2_npiv)
            evs[q][1].record()
            tab2_npiv += 1
        torch.cuda.synchronize()
        # the first launches pay CUDA's lazy module load of kernels the fused loop never used: drop them
        upd_ms = statistics.mean(a.elapsed_time(b) for a, b in evs[5:])
        pick_ms = statistics.mean(a.elapsed_time(b) for a, b in pick_evs[5:])
        k3 = alg_bytes / (upd_ms * 1e-3) / 1e9
        k3_traffic = None
        if os.path.exists(tp):
            with open(tp) as fh:
                k3_traffic = json.load(fh).get("dram_bytes_per_launch")
        roofline_k3 = {"bound": "hbm", "kernel": "update_tiled_kernel (K3: one pivot per pass, 16 B per cell per pivot)",
                       "achieved": k3, "peak": peak, "unit": "GB/s", "frac": k3 / peak, "traffic": k3_traffic,
                       "algorithmic_bytes_per_launch": alg_bytes, "update_ms": upd_ms, "pick_ms": pick_ms,
                       "frac_of_nominal_8TBs": k3 / 8000.0}
        del tab
        torch.cuda.empty_cache()

        # ---------------- e2e: public API, pinned host input, upload inside the timed region
        pinned = torch.empty((N_ROWS, M_COLS + 1), dtype=torch.float64).pin_memory()
        pinned.numpy()[...] = rows
        host_rows = pinned.numpy()
        h2d = host_rows.nbytes + c.nbytes
        e2e_steps = max(1, min(args.steps, 3))
        e2e_t, d2h = [], 0
        for it in range(1 + e2e_steps):            # first iteration is a warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sm = SimplexMethod(host_rows, c, device=dev, engine="stream")
            sol = sm.solve(max_pivots=P, chunk=P)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            assert sol.npiv == P and (sol.trace == gold[:P]).all()
            d2h = sol.trace.nbytes + sol.x.nbytes + 16 + sol.rowlab.nbytes + sol.collab.nbytes
            if it > 0:
                e2e_t.append(dt)
            del sm
        e2e_val = P / statistics.mean(e2e_t)
        del pinned, host_rows
        torch.cuda.empty_cache()

        cpu = cpu_baseline_sample(rows, c, gold) if not args.no_cpu_baseline else None
        del rows
        batched = batched_big = resident = cfg1 = cfg5 = None
        if not args.no_batched:
            batched = batched_leg(dev, 0, 1)
            batched_big = batched_leg(dev, 0, 1, reps=6, B=1 << 20, golden=False)
            resident = resident_leg(dev)
            cfg1, cfg5 = small_legs(dev)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(), "implementation": implementation_dict(1), "clocks": clk.summary(),
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": 1e3 * statistics.mean(e2e_t),
                    "api": f"SimplexMethod(pinned_rows, c).solve(max_pivots={P})"},
            "gpu_launches": launches, "roofline": roofline, "roofline_single_pivot_kernel": roofline_k3,
            "cpu_baseline": cpu, "cpu_baseline_reference": python_reference_timings() if not args.no_cpu_baseline else None,
            "northstar_convention_GBps_whole_step": alg_bytes * args.steps * P / (total_ms * 1e-3) / 1e9,
            "batched": batched, "batched_1M": batched_big, "l2_resident": resident, "cfg1_gui_lp": cfg1,
            "cfg5_klee_minty_20": cfg5,
            "parity": parity,
        }
        print(json.dumps(line), flush=True)
        return

    # ---------------- N > 1: column-sharded, one process per GPU ---------------------------
    from simplex_method_solver_b200.parallel import FusedShardedTableau, PeerShardedTableau, ShardedTableau
    fallback_note = None
    owner_changes = None
    price_engine = None
    if args.exchange == "fused":
        # passes of 8 pivots: cooperative pricing with the in-kernel NVLink exchange, then ONE stream
        # over the local columns applies them all (csrc/spx_fused.cu).  If peer memory cannot be mapped on
        # this box (no CUDA IPC / P2P between the GPUs) every rank falls back to the NCCL all-gather flow.
        # Pricing engines to try, in order: the per-pass engine (one pricing kernel per pass, the default) or, on
        # request, the persistent engine first (one pricing kernel per run() call, device-flag hand-shakes with the
        # update kernels).  Each goes through the same two preflights before it may be timed.
        if args.no_lookahead:
            engines = [False]
        elif args.price_engine == "auto":
            engines = (["persistent", "per-pass"] if 0 < FusedShardedTableau.PERSISTENT_FROM_WORLD <= world
                       else ["per-pass"])
        else:
            engines = [args.price_engine] + (["per-pass"] if args.price_engine == "persistent" else [])
        sh, peer_memory_ok, notes = None, True, []
        for engine in engines:
            sh, err = None, ""
            try:
                sh = FusedShardedTableau(N_ROWS, M_COLS, rank, world, device=dev, trace_capacity=need + 64,
                                         depth=args.depth or fused_depth_for(world), lookahead=engine)
            except Exception as e:                   # noqa: BLE001 - reported below, then the documented fallback
                err = f"{type(e).__name__}: {e}"
            okf = torch.tensor([1 if sh is not None else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
            if int(okf.item()) == 0:
                log(f"[rank {rank}] peer-memory exchange unavailable ({err or 'a peer failed'}); falling back to --exchange nccl")
                notes.append(f"peer memory unavailable ({err or 'on a peer'})")
                if sh is not None:
                    sh.close()
                sh, peer_memory_ok = None, False
                break
            # preflight 1: the committed "late" LP — entering columns owned by every rank, > 100 owner changes —
            # full table against the oracle's golden; preflight 2: a few passes of cfg4 against the golden prefix.
            # A rank that times out on a peer (SPX_PEER_TIMEOUT) or diverges sends all ranks to the next engine and,
            # after the last one, to the pivot-at-a-time peer-mailbox loop (csrc/spx_shard.cu); the printed line says so
            ok_late, owner_changes, why = late_lp_preflight(
                lambda *a_, **k_: FusedShardedTableau(*a_, lookahead=engine, **k_), rank, world, dev, dist)
            pre = 96
            if ok_late:
                try:
                    sh.load(rows, c, max_pivots=pre + 64)
                    sh.run(pre)
                    stp = sh.sync()
                    trp = sh.trace[:pre].cpu().numpy()
                    if stp.status != N.PIVOT or stp.npiv != pre:
                        why = f"status {stp.status} after {stp.npiv} pivots"
                    elif not (trp == gold[:pre]).all():
                        why = "pivot sequence differs from the golden prefix"
                except Exception as e:                   # noqa: BLE001
                    why = f"{type(e).__name__}: {e}"
            okf = torch.tensor([0 if why else 1], dtype=torch.int32, device=dev)
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
            if int(okf.item()) == 1:
                price_engine = {False: "none (no look-ahead)"}.get(engine, engine)
                break
            log(f"[rank {rank}] fused exchange, pricing engine {engine!r}, failed its preflight ({why or 'on a peer'})")
            notes.append(f"fused preflight failed with pricing engine {engine!r} ({why or 'on a peer'})")
            sh.close()
            sh = None
        if sh is None and not peer_memory_ok:
            args.exchange = "nccl"
            sh = ShardedTableau(N_ROWS, M_COLS, rank, world, device=dev, trace_capacity=need + 64,
                                lookahead=not args.no_lookahead)
        elif sh is None:
            log(f"[rank {rank}] falling back to --exchange p2p")
            args.exchange = "p2p"
            sh = PeerShardedTableau(N_ROWS, M_COLS, rank, world, device=dev, trace_capacity=need + 64)
        fallback_note = "; ".join(notes) or None
    elif args.exchange == "p2p":
        # C-side look-ahead loop, candidates exchanged by NVLink peer stores (csrc/spx_shard.cu)
        sh = PeerShardedTableau(N_ROWS, M_COLS, rank, world, device=dev, trace_capacity=need + 64)
    else:
        sh = ShardedTableau(N_ROWS, M_COLS, rank, world, device=dev, trace_capacity=need + 64,
                            lookahead=not args.no_lookahead)
    sh.load(rows, c, max_pivots=need + 64)
    for _ in range(args.warmup):
        sh.run(P)
    torch.cuda.synchronize()
    dist.barrier()
    N.load().spx_launch_count(1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        torch.cuda.synchronize()
        dist.barrier()
        ev0.record()
        for _ in range(args.steps):
            sh.run(P)
        ev1.record()
        torch.cuda.synchronize()
        dist.barrier()
    launches = int(N.load().spx_launch_count(0))
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    st = sh.sync()
    assert st.npiv == need and st.status == N.PIVOT, (st.status, st.npiv)
    tr = sh.trace[:need].cpu().numpy()

    def table_digests():
        """b (replicated) and, all-reduced over the ranks' column blocks, the f row sha256 and the body checksum."""
        if args.exchange == "fused":
            body, bcur = sh.local_body(), sh.b_current()
        else:
            cur = int(st.npiv) & 1
            body, bcur = sh.A[cur, :, : sh.m_loc], sh.b[cur, :N_ROWS]
        ck = torch.tensor([as_i64(W.body_checksum_torch(body[:N_ROWS], m_total=M_COLS, col0=sh.col0)) if sh.m_loc else 0],
                          dtype=torch.int64, device=dev)
        dist.all_reduce(ck)
        fs = [None] * world
        dist.all_gather_object(fs, body[N_ROWS].cpu().numpy().tobytes())
        return (hashlib.sha256(bcur.cpu().numpy().tobytes()).hexdigest(), hashlib.sha256(b"".join(fs)).hexdigest(),
                int(ck.item()) & 0xFFFFFFFFFFFFFFFF)

    pricing_levels = None
    if args.exchange == "fused" and rank == 0:
        # per-level phase breakdown of the LAST pricing kernel of the timed region (%globaltimer stamps, rank 0)
        stp = sh.pricing_stamps().astype(np.int64)
        dep = args.depth or fused_depth_for(world)
        lv = stp[1:dep]                                  # levels 1..depth-1 of the pass: all six stamps are from this launch
        d = np.diff(np.concatenate([stp[0:dep - 1, 5:6], lv], axis=1), axis=1) / 1e3
        pricing_levels = {"us_per_level": float((stp[dep - 1, 5] - stp[0, 5]) / ((dep - 1) * 1e3)),
                          "phases_us_mean": {k: float(v) for k, v in zip(
                              ["phase_A_b_f_row_replay", "grid_barrier_entering_column", "candidate_column_build_and_store",
                               "arrive_nvlink_key_exchange_broadcast", "ratio_fold_grid_barrier", "final_merge_and_record"],
                              d.mean(axis=0))},
                          "how": f"%globaltimer stamps by thread 0 of rank 0 in shard_price_kernel, last pass, levels 1-{dep - 1}"}
    parity = "sharded " + check_against_marks(tr, need, marks, gold, table_digests)
    value = args.steps * P / (total_ms * 1e-3)
    alg_bytes = 16.0 * cells(N_ROWS, M_COLS)

    # ---------------- e2e at N GPUs: every rank uploads ITS column block from pinned host memory, the
    # ranks pivot together, every rank reads its state and trace back; wall clock between barriers, max over ranks
    e2e = None
    if args.exchange in ("fused", "p2p"):
        blk = torch.empty((N_ROWS, sh.m_loc + 1), dtype=torch.float64).pin_memory()
        blk.numpy()[:, : sh.m_loc] = rows[:, sh.col0: sh.col0 + sh.m_loc]
        blk.numpy()[:, sh.m_loc] = rows[:, M_COLS]
        cblk = np.ascontiguousarray(c[sh.col0: sh.col0 + sh.m_loc])
        e2e_steps = max(1, min(args.steps, 3))
        ts = []
        for it in range(1 + e2e_steps):                     # first iteration is a warm-up
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            sh.load_local(blk.numpy(), cblk, max_pivots=P + 64)
            sh.run(P)
            st2 = sh.sync()
            tr2 = sh.trace[:P].cpu().numpy()
            torch.cuda.synchronize()
            dist.barrier()
            dt = time.perf_counter() - t0
            assert st2.npiv == P and (tr2 == gold[:P]).all(), "e2e: sharded pivot sequence differs from the golden prefix"
            if it > 0:
                ts.append(dt)
        tmax = torch.tensor([statistics.mean(ts)], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e = {"value": P / float(tmax.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(8 * (N_ROWS * (M_COLS + world) + M_COLS)),
               "d2h_bytes_per_step": int(world * (tr2.nbytes + 128)), "steps": e2e_steps,
               "ms_per_step": 1e3 * float(tmax.item()),
               "api": f"{type(sh).__name__}.load_local(pinned_block, c_block); run({P}); sync() on every rank"}
        del blk
    del rows
    batched = batched_big = None
    if not args.no_batched:
        batched = batched_leg(dev, rank, world, dist)
        batched_big = batched_leg(dev, rank, world, dist, reps=6, B=1 << 20, golden=False)
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(),
            "implementation": implementation_dict(world, args.exchange, fallback_note,
                                                  price_engine if args.exchange == "fused" else None),
            "clocks": clk.summary(),
            "e2e": e2e, "gpu_launches": launches,
            "roofline": {"bound": "hbm",
                         "kernel": ("update_lazy_kernel (K6)" if args.exchange == "fused" else "update_tiled_kernel (K3)") +
                                   ": WHOLE step incl. pricing and exchange, 16 B x cells per pivot / step time / N",
                         "achieved": alg_bytes * args.steps * P / (total_ms * 1e-3) / 1e9 / world,
                         "peak": peak, "unit": "GB/s per GPU", "peak_source": peak_src,
                         "frac": alg_bytes * args.steps * P / (total_ms * 1e-3) / 1e9 / world / peak,
                         "traffic": None},
            "cpu_baseline": None, "batched": batched, "batched_1M": batched_big,
            "pricing_level_breakdown": pricing_levels,
            "parity": parity,
            "parity_owner_changes": owner_changes,
            "parity_late_lp": (None if owner_changes is None else
                               f"late LP (tests/golden/late_lp.json) through the fused sharded loop on {world} ranks: trace, b, "
                               f"f and body checksum == oracle golden; the entering column changed owner rank {owner_changes} times"
                               if args.exchange == "fused" else "FAILED: " + str(fallback_note)),
        }
        print(json.dumps(line), flush=True)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-pivots-per-step", type=int, default=4)
    ap.add_argument("--python-reference-only", action="store_true",
                    help="--impl reference: only time the reference's own simplex.py ($SIMPLEX_REF) and print that")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batched", action="store_true", help="skip the cfg1/cfg2/cfg3/cfg5 legs")
    ap.add_argument("--depth", type=int, default=0, help="N>1 fused loop: pivots per pass (0 = default)")
    ap.add_argument("--exchange", default="fused", choices=["fused", "p2p", "nccl"],
                    help="N>1: fused passes with the in-kernel NVLink exchange (default); pivot-at-a-time look-ahead "
                         "with NVLink peer mailboxes (p2p) or an NCCL all-gather (nccl)")
    ap.add_argument("--shard-threads", type=int, default=0,
                    help="N>1 fused loop: threads per CTA of the sharded pricing kernel (0 = library default)")
    ap.add_argument("--shard-ctas", type=int, default=0,
                    help="N>1 fused loop: cap on the CTAs (= SMs) of the sharded pricing kernel (0 = library default)")
    ap.add_argument("--price-engine", default="auto", choices=["auto", "persistent", "per-pass"],
                    help="N>1 fused loop: pricing engine (auto = one pricing kernel per pass; persistent = one per run() call, "
                         "measured no faster: profiles/r2/r2q_r2r_persistent_engine.md)")
    ap.add_argument("--no-lookahead", action="store_true",
                    help="classic pick->update order instead of pricing pivot k+1 during update k")
    ap.add_argument("--max-connections", type=int, default=0,
                    help="CUDA_DEVICE_MAX_CONNECTIONS for this process (hardware work queues the streams share; the CUDA "
                         "default is 8); 0 = leave the environment alone.  Must be set before CUDA initialises.")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last step computed to DIR/<name>.npy (float64): its "
                         "pivots, b, the f row, x, objective, labels and a seeded sample of the body cells")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs covers the single-GPU timed loop (--impl ours --gpus 1)")
    if args.max_connections > 0:
        os.environ["CUDA_DEVICE_MAX_CONNECTIONS"] = str(args.max_connections)
    if args.warmup < 3 and args.impl == "ours":
        log("note: the timing rules ask for >= 3 warm-up steps")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
