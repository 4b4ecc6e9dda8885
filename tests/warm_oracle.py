"""Loader of warm_oracle.c (the sequential statement of the change of final tables) and the resume of one LP by the
pinned oracle's own loop — test infrastructure only.

The C file is compiled once per process into a temporary directory, so a read-only checkout works.  ``resume`` calls
``orc_solve_rule`` of oracle/spx_oracle.c with the given labels (it never initialises them) and ``orc_extract`` with
the given costs, so a resumed LP is checked by the same code as a fresh one.
"""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="spx_warm_oracle_")
        so = os.path.join(d, "libwarm.so")
        cc = shutil.which("gcc") or shutil.which("cc") or "/usr/bin/gcc"
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-o", so,
                        os.path.join(HERE, "warm_oracle.c")], check=True, capture_output=True)
        L = ctypes.CDLL(so)
        dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int32)
        L.orc_warm_change.argtypes = [dp, ctypes.c_int, ctypes.c_int, ip, ip, dp, dp]
        L.orc_warm_change.restype = None
        _lib = L
    return _lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _ip(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))


def change(T, n: int, m: int, rowlab, collab, db=None, dc=None) -> np.ndarray:
    """One LP's changed table (a new array)."""
    T = np.array(T, dtype=np.float64, copy=True).reshape(-1)
    rl = np.ascontiguousarray(rowlab, dtype=np.int32).reshape(-1)
    cl = np.ascontiguousarray(collab, dtype=np.int32).reshape(-1)
    assert T.shape[0] == n * (m + 1) + m and rl.shape[0] == m and cl.shape[0] == n
    db = None if db is None else np.ascontiguousarray(db, dtype=np.float64).reshape(n)
    dc = None if dc is None else np.ascontiguousarray(dc, dtype=np.float64).reshape(m)
    lib().orc_warm_change(_dp(T), n, m, _ip(rl), _ip(cl), _dp(db), _dp(dc))
    return T


def resume(T, n: int, m: int, rowlab, collab, function, max_pivots: int, rule: str = "reference",
           snapshots: bool = False) -> oracle.Solve:
    """Continue one LP from table T and labels (rowlab, collab) for up to max_pivots pivots; obj2 / objm use
    `function`, the LP's current costs."""
    T = np.array(T, dtype=np.float64, copy=True).reshape(-1)
    cells = n * (m + 1) + m
    rl = np.array(rowlab, dtype=np.int32, copy=True).reshape(-1)
    cl = np.array(collab, dtype=np.int32, copy=True).reshape(-1)
    fn = np.ascontiguousarray(function, dtype=np.float64).reshape(m)
    scratch = np.empty(cells)
    trace = np.zeros((max(max_pivots, 1), 2), dtype=np.int32)
    snaps = np.empty((max_pivots + 1, cells)) if snapshots else None
    npiv = ctypes.c_int64(0)
    L = oracle.lib()
    st = L.orc_solve_rule(oracle._dp(T), oracle._dp(scratch), n, m, oracle.RULES[rule], max_pivots,
                          oracle._ip(trace), oracle._dp(snaps), oracle._ip(rl), oracle._ip(cl), ctypes.byref(npiv))
    k = npiv.value
    x = np.zeros(m)
    o2, om = ctypes.c_double(0.0), ctypes.c_double(0.0)
    L.orc_extract(oracle._dp(T), n, m, oracle._ip(cl), oracle._dp(fn), oracle._dp(x), ctypes.byref(o2),
                  ctypes.byref(om))
    return oracle.Solve(st, k, trace[:k].copy(), T, rl, cl, x, o2.value, om.value,
                        snaps[: k + 1].copy() if snapshots else None)
