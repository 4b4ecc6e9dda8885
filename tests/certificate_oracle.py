"""The certificate report's sequential statement (spx_certificate_*, include/spx_b200.h) — test infrastructure only.

``certificate`` runs certificate_oracle.c, compiled once per process into a temporary directory (so a read-only
checkout works).  ``py_certificate`` is the same statement written again in plain Python floats, independently of the
C file; the tests check the two against each other.
"""
import ctypes
import math
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
        d = tempfile.mkdtemp(prefix="spx_cert_oracle_")
        so = os.path.join(d, "libcert.so")
        cc = shutil.which("gcc") or shutil.which("cc") or "/usr/bin/gcc"
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-o", so,
                        os.path.join(HERE, "certificate_oracle.c"), "-lm"], check=True, capture_output=True)
        L = ctypes.CDLL(so)
        dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int32)
        L.orc_certificate.argtypes = [dp, ctypes.c_int, ctypes.c_int, ip, ip, ip, dp, dp, ip, dp, dp]
        L.orc_certificate.restype = None
        _lib = L
    return _lib


def certificate(T, n: int, m: int, rowlab, collab):
    """One LP's report: (farkas_row, farkas [n], farkas_bound, ray_col, ray [m], ray_slope)."""
    T = np.ascontiguousarray(T, dtype=np.float64).reshape(-1)
    rl = np.ascontiguousarray(rowlab, dtype=np.int32).reshape(-1)
    cl = np.ascontiguousarray(collab, dtype=np.int32).reshape(-1)
    assert T.shape[0] == n * (m + 1) + m and rl.shape[0] == m and cl.shape[0] == n
    row, col = np.zeros(1, np.int32), np.zeros(1, np.int32)
    farkas, ray, bound, slope = np.empty(n), np.empty(m), np.empty(1), np.empty(1)
    dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
    ip = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))  # noqa: E731
    lib().orc_certificate(dp(T), n, m, ip(rl), ip(cl), ip(row), dp(farkas), dp(bound), ip(col), dp(ray), dp(slope))
    return int(row[0]), farkas, float(bound[0]), int(col[0]), ray, float(slope[0])


def py_certificate(T, n: int, m: int, rowlab, collab):
    """The same statement in plain Python floats: (farkas_row, farkas, farkas_bound, ray_col, ray, ray_slope)."""
    T = [float(v) for v in np.asarray(T, dtype=np.float64).reshape(-1)]
    rowlab = [int(v) for v in np.asarray(rowlab).reshape(-1)]
    collab = [int(v) for v in np.asarray(collab).reshape(-1)]
    w = m + 1
    cell = lambda i, j: T[i * w + j]  # noqa: E731
    b = [cell(i, m) for i in range(n)]
    d = T[n * w:]
    fin = math.isfinite
    nan = float("nan")

    r = next((i for i in range(n) if fin(b[i]) and b[i] < 0 and all(fin(cell(i, j)) and cell(i, j) <= 0
                                                                   for j in range(m))), -1)
    farkas, bound = [nan] * n, nan
    if r >= 0:
        farkas = [0.0] * n
        if m <= collab[r] < m + n:
            farkas[collab[r] - m] = 1.0
        for j in range(m):
            if m <= rowlab[j] < m + n:
                farkas[rowlab[j] - m] = 0.0 - cell(r, j)
        bound = b[r]

    c = -1
    if all(fin(v) and v >= 0 for v in b):
        c = next((j for j in range(m) if fin(d[j]) and d[j] < 0 and all(fin(cell(i, j)) and cell(i, j) >= 0
                                                                       for i in range(n))), -1)
    ray, slope = [nan] * m, nan
    if c >= 0:
        ray = [0.0] * m
        if 0 <= rowlab[c] < m:
            ray[rowlab[c]] = 1.0
        for i in range(n):
            if 0 <= collab[i] < m:
                ray[collab[i]] = cell(i, c) + 0.0
        slope = d[c]
    return r, np.asarray(farkas, dtype=np.float64), bound, c, np.asarray(ray, dtype=np.float64), slope
