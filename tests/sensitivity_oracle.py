"""Loader of sensitivity_oracle.c (the sequential statement of the sensitivity report) — test infrastructure only.

The C file is compiled once per process into a temporary directory, so a read-only checkout works.
"""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="spx_sens_oracle_")
        so = os.path.join(d, "libsens.so")
        cc = shutil.which("gcc") or shutil.which("cc") or "/usr/bin/gcc"
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-o", so,
                        os.path.join(HERE, "sensitivity_oracle.c"), "-lm"], check=True, capture_output=True)
        L = ctypes.CDLL(so)
        dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int32)
        L.orc_sensitivity.argtypes = [dp, ctypes.c_int, ctypes.c_int, ip, ip, ctypes.c_int, dp, dp, dp, dp, dp]
        L.orc_sensitivity.restype = None
        _lib = L
    return _lib


def sensitivity(T, n: int, m: int, rowlab, collab, optimal: bool):
    """One LP's report: (dual [n], slack [n], reduced_cost [m], rhs_range [n, 2], cost_range [m, 2])."""
    T = np.ascontiguousarray(T, dtype=np.float64).reshape(-1)
    rl = np.ascontiguousarray(rowlab, dtype=np.int32).reshape(-1)
    cl = np.ascontiguousarray(collab, dtype=np.int32).reshape(-1)
    assert T.shape[0] == n * (m + 1) + m and rl.shape[0] == m and cl.shape[0] == n
    out = [np.empty(n), np.empty(n), np.empty(m), np.empty((n, 2)), np.empty((m, 2))]
    dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
    ip = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))  # noqa: E731
    lib().orc_sensitivity(dp(T), n, m, ip(rl), ip(cl), int(bool(optimal)), *[dp(a) for a in out])
    return tuple(out)
