"""Loader of dantzig_bland_oracle.c (the sequential statement of Dantzig's rule with Bland's rule on degenerate pivots
and a ratio-tested phase 1, SPX_RULE_DANTZIG_BLAND) — test infrastructure only.

dantzig_bland_oracle.c is compiled together with oracle/spx_oracle.c, once per process into a temporary directory (a
read-only checkout works), so the pivot, the labels and the extraction are the pinned oracle's own code.
"""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="spx_db_oracle_")
        so = os.path.join(d, "libdb.so")
        cc = shutil.which("gcc") or shutil.which("cc") or "/usr/bin/gcc"
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-o", so,
                        os.path.join(HERE, "dantzig_bland_oracle.c"), os.path.join(ROOT, "oracle", "spx_oracle.c")],
                       check=True, capture_output=True)
        L = ctypes.CDLL(so)
        dp, ip, i64 = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int32), ctypes.c_int64
        pint = ctypes.POINTER(ctypes.c_int)
        L.orc_pick_db.argtypes = [dp, ctypes.c_int, ctypes.c_int, ip, ip, pint, pint]
        L.orc_pick_db.restype = ctypes.c_int
        L.orc_solve_db.argtypes = [dp, dp, ctypes.c_int, ctypes.c_int, i64, ip, dp, ip, ip, ctypes.POINTER(i64)]
        L.orc_solve_db.restype = ctypes.c_int
        L.orc_extract.argtypes = [dp, ctypes.c_int, ctypes.c_int, ip, dp, dp, dp, dp]
        L.orc_extract.restype = None
        _lib = L
    return _lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _ip(a):
    return None if a is None else a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))


def pick(T, n: int, m: int, rowlab=None, collab=None):
    """(status, r, c) of one pick on reference-flat T with the given labels (default 'x1'.. / 'y1'..)"""
    T = np.ascontiguousarray(T, dtype=np.float64)
    rl0, cl0 = oracle.init_labels(n, m)
    rl = rl0 if rowlab is None else np.ascontiguousarray(rowlab, dtype=np.int32)
    cl = cl0 if collab is None else np.ascontiguousarray(collab, dtype=np.int32)
    r, c = ctypes.c_int(-1), ctypes.c_int(-1)
    st = lib().orc_pick_db(_dp(T), n, m, _ip(rl), _ip(cl), ctypes.byref(r), ctypes.byref(c))
    return st, r.value, c.value


def solve_flat(T0, n: int, m: int, max_pivots: int = 1_000_000, snapshots: bool = False, rowlab=None,
               collab=None, function=None) -> oracle.Solve:
    """A solve of reference-flat T0 under the rule.  Fresh (labels None): labels 'x1'.. / 'y1'.., obj from
    T0's f row.  Resume: from the given labels, obj from `function` (the LP's current costs)."""
    T = np.array(T0, dtype=np.float64, copy=True).reshape(-1)
    cells = n * (m + 1) + m
    assert T.shape[0] == cells
    if rowlab is None:
        rl, cl = oracle.init_labels(n, m)
    else:
        rl = np.array(rowlab, dtype=np.int32, copy=True).reshape(-1)
        cl = np.array(collab, dtype=np.int32, copy=True).reshape(-1)
    fn = T[n * (m + 1):].copy() if function is None else np.ascontiguousarray(function, dtype=np.float64).reshape(m)
    scratch = np.empty(cells)
    trace = np.zeros((max(max_pivots, 1), 2), dtype=np.int32)
    snaps = np.empty((max_pivots + 1, cells)) if snapshots else None
    npiv = ctypes.c_int64(0)
    L = lib()
    st = L.orc_solve_db(_dp(T), _dp(scratch), n, m, max_pivots, _ip(trace), _dp(snaps), _ip(rl), _ip(cl),
                           ctypes.byref(npiv))
    k = npiv.value
    x = np.zeros(m)
    o2, om = ctypes.c_double(0.0), ctypes.c_double(0.0)
    L.orc_extract(_dp(T), n, m, _ip(cl), _dp(fn), _dp(x), ctypes.byref(o2), ctypes.byref(om))
    return oracle.Solve(st, k, trace[:k].copy(), T, rl, cl, x, o2.value, om.value,
                        snaps[: k + 1].copy() if snapshots else None)


def solve(constraints, function, max_pivots: int = 1_000_000, snapshots: bool = False) -> oracle.Solve:
    T, n, m = oracle.flatten(constraints, function)
    return solve_flat(T, n, m, max_pivots, snapshots)
