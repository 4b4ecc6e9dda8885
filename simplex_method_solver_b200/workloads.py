"""Synthetic LP generators and digest conventions for the five BASELINE.json configs.

These are measurement-input specifications (SURVEY.md §8d / Appendix A), not
solver code: numpy 2.x ``default_rng`` (PCG64), fixed draw order.  Every LP is
in the reference's input convention (``SimplexMethod(constraints, function)``,
/root/reference/src/simplex.py:25): row i of ``constraints`` is
``[a_i1..a_im, b_i]`` meaning ``a_i.x + b_i >= 0``, and ``function`` is
minimised.
"""
from __future__ import annotations

import hashlib
import struct

import numpy as np


def dense_lp(n: int, m: int, seed: int = 0):
    """D(n, m, seed): dense, origin-feasible, bounded (cfg2: 1000x2000, cfg4: 16384x32768).

    Returns (rows [n, m+1] fp64, c [m] fp64).
    """
    g = np.random.default_rng(seed)
    rows = np.empty((n, m + 1), dtype=np.float64)
    # draw order A, b, c — written straight into the [A | b] matrix so cfg4 never
    # holds two 4.3 GB copies
    rows[:, :m] = g.uniform(0.1, 1.0, (n, m))
    np.negative(rows[:, :m], out=rows[:, :m])
    rows[:, m] = g.uniform(1.0, 2.0, n) * m
    c = -g.uniform(0.1, 1.0, m)
    return rows, c


def phase1_lp(n: int, m: int, seed: int = 0):
    """D(n, m, seed) pushed into phase 1: a tenth of the rows (at least one) get a negated and
    b = -b * U(0.05, 0.2) (origin infeasible, simplex.py:72-91), and 5 % of the a cells are exact zeros.
    Ends OPTIMAL after a few hundred to a few thousand pivots at the sizes of tools/cluster_bench.py.

    Returns (rows [n, m+1] fp64, c [m] fp64).
    """
    rows, c = dense_lp(n, m, seed)
    g = np.random.default_rng([seed, 1])
    idx = g.choice(n, max(1, n // 10), replace=False)
    rows[idx, :m] = -rows[idx, :m]
    rows[idx, m] = -rows[idx, m] * g.uniform(0.05, 0.2, idx.shape[0])
    body = rows[:, :m]
    body[g.random((n, m)) < 0.05] = 0.0
    return rows, c


def gui_batch(B: int, seed: int = 0):
    """P(B, seed): GUI-like 8-constraint / 2-variable LPs (cfg3: B=65536).

    Bounded octagon around (5, 5), origin infeasible (exercises the phase-1
    branch, simplex.py:72-91), coefficients rounded to 2 dp as the GUI does
    (plot_widget.py:408).  Returns (T [B, 8, 3], C [B, 2]).
    """
    g = np.random.default_rng(seed)
    k = np.arange(8)[None, :]
    th = 2 * np.pi * (k + g.uniform(0, 1, (B, 8))) / 8
    nx, ny = -np.cos(th), -np.sin(th)
    r = g.uniform(1.0, 4.0, (B, 8))
    p0 = 5.0
    T = np.round(np.stack([nx, ny, r - (nx * p0 + ny * p0)], axis=2), 2)
    ph = g.uniform(0, 2 * np.pi, B)
    C = np.round(np.stack([np.cos(ph), np.sin(ph)], axis=1), 2)
    return T, C


def gui_ragged(B: int, seed: int = 0):
    """GUI-like bounded polygons of 3 to 12 sides (k constraints, 2 variables): gui_batch's octagon construction with
    the number of sides drawn per LP.  Returns a list of B (rows [k, 3], c [2]) pairs (10 shapes, all <= 38 cells)."""
    g = np.random.default_rng([seed, 3])
    sides = g.integers(3, 13, B)
    out = []
    for k in sides:
        k = int(k)
        th = 2 * np.pi * (np.arange(k) + g.uniform(0, 1, k)) / k
        nx, ny = -np.cos(th), -np.sin(th)
        r = g.uniform(1.0, 4.0, k)
        p0 = 5.0
        rows = np.round(np.stack([nx, ny, r - (nx * p0 + ny * p0)], axis=1), 2)
        ph = g.uniform(0, 2 * np.pi)
        out.append((rows, np.round(np.array([np.cos(ph), np.sin(ph)]), 2)))
    return out


def mixed_lps(B: int, seed: int = 0):
    """B LPs of the dense and phase-1 families with n and m drawn log-uniformly from geometric grids of 24 values,
    1..512 and 2..800 (a few hundred shapes), so they spread over K4 warp mode (<= 96 cells), K4 CTA mode
    (<= 10,000 cells) and K7 at every cluster size; every shape fits one cluster (n <= 528 at m = 800).
    Returns a list of B (rows [n, m+1], c [m]) pairs."""
    g = np.random.default_rng([seed, 5])
    ns = np.unique(np.round(np.geomspace(1, 512, 24)).astype(int))
    ms = np.unique(np.round(np.geomspace(2, 800, 24)).astype(int))
    out = []
    for k in range(B):
        n, m = int(g.choice(ns)), int(g.choice(ms))
        fam = phase1_lp if g.random() < 0.5 else dense_lp
        out.append(fam(n, m, seed * 1_000_003 + k))
    return out


def scaled_lps(B: int, seed: int = 0):
    """mixed_lps(B, seed) with the units of every x_j changed: column j of the constraints and c_j multiplied by
    10^U(-2, 2) (draws from seed + 7, one per column of each LP in turn).  The same LPs up to scale, so the pivot counts
    of the scale-dependent entering rules (reference, Dantzig) and of devex can be compared on badly scaled inputs.
    Returns a list of B (rows [n, m+1], c [m]) pairs."""
    g = np.random.default_rng(seed + 7)
    out = []
    for rows, c in mixed_lps(B, seed):
        s = 10.0 ** g.uniform(-2.0, 2.0, c.shape[0])
        rows[:, : c.shape[0]] *= s
        out.append((rows, c * s))
    return out


def mixed_large_lps(B: int = 1024, seed: int = 0):
    """mixed_lps(B, seed) with cap 20,000 each, then 32 LPs above K7's capacity with cap 4,000 each: 8 each of
    D(600, 800), phase-1 1000 x 1000, D(2000, 300) and D(64, 12000), in that order (seeds seed * 1_000_003 + B + q
    for the q-th of them).  Every K4 class, every K7 cluster size and two K8 launches (S_min 1, and S_min 2 for
    64 x 12000).  Returns (lps, caps): a list of B + 32 (rows [n, m+1], c [m]) pairs and the list of their caps."""
    lps = mixed_lps(B, seed)
    caps = [20000] * len(lps)
    large = [(dense_lp, 600, 800), (phase1_lp, 1000, 1000), (dense_lp, 2000, 300), (dense_lp, 64, 12000)]
    q = 0
    for fam, n, m in large:
        for _ in range(8):
            lps.append(fam(n, m, seed * 1_000_003 + B + q))
            caps.append(4000)
            q += 1
    return lps, caps


def klee_minty(n: int):
    """KM(n): Klee-Minty cube, all floats (cfg5: n=20, 2^n - 1 pivots)."""
    rows = []
    for i in range(1, n + 1):
        r = [0.0] * (n + 1)
        for j in range(1, i):
            r[j - 1] = -float(2 ** (i - j + 1))
        r[i - 1] = -1.0
        r[n] = float(5 ** i)
        rows.append(r)
    c = [-float(2 ** (n - j)) for j in range(1, n + 1)]
    return np.asarray(rows, dtype=np.float64), np.asarray(c, dtype=np.float64)


# the reference's own cfg1 example, simplex.py:205-209
CFG1_ROWS = [[-39.70, -96.00, 4060.80],
             [-45.50, 45.30, 600.60],
             [45.50, -7.40, -54.60],
             [24.20, 45.10, -1091.42]]
CFG1_C = [-1.0, -1.0]


def batch_flat(T: np.ndarray, C: np.ndarray) -> np.ndarray:
    """[B, n, m+1] rows + [B, m] functions -> [B, cells] reference-flat tables."""
    B = T.shape[0]
    return np.ascontiguousarray(np.concatenate([T.reshape(B, -1), C.reshape(B, -1)], axis=1),
                                dtype=np.float64)


def input_digest(rows: np.ndarray, c: np.ndarray) -> str:
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(rows).astype("<f8", copy=False).tobytes())
    h.update(np.ascontiguousarray(c).astype("<f8", copy=False).tobytes())
    return h.hexdigest()


def pivot_digest(trace) -> str:
    """sha256 over '<ii' (r, c) per pivot, in order (single LP)."""
    t = np.ascontiguousarray(np.asarray(trace, dtype="<i4").reshape(-1, 2))
    return hashlib.sha256(t.tobytes()).hexdigest()


def batch_pivot_digest(trace: np.ndarray, npiv: np.ndarray) -> str:
    """sha256 over '<iii' (k, r, c) for LP k in order, each pivot in order."""
    B = trace.shape[0]
    npiv = np.asarray(npiv).astype(np.int64)
    kk = np.repeat(np.arange(B, dtype=np.int64), npiv)
    pos = np.arange(int(npiv.sum()), dtype=np.int64) - np.repeat(np.cumsum(npiv) - npiv, npiv)
    rc = np.asarray(trace)[kk, pos]
    rec = np.empty((kk.shape[0], 3), dtype="<i4")
    rec[:, 0] = kk
    rec[:, 1:] = rc
    return hashlib.sha256(rec.tobytes()).hexdigest()


def batch_solution_digest(x1, x2, f) -> str:
    """sha256 over '<ddd' (x1, x2, f) per LP."""
    rec = np.stack([np.asarray(x1, dtype="<f8"), np.asarray(x2, dtype="<f8"),
                    np.asarray(f, dtype="<f8")], axis=1)
    return hashlib.sha256(np.ascontiguousarray(rec).tobytes()).hexdigest()


def snapshot_digest(tables) -> str:
    """sha256 over every cell of every snapshot table, '<d', row-major."""
    h = hashlib.sha256()
    for tab in tables:
        for row in tab:
            for v in row:
                h.update(struct.pack("<d", float(v)))
    return h.hexdigest()


def body_checksum_numpy(body: np.ndarray) -> int:
    """Order-free 64-bit checksum of an [n, m] fp64 body (a strided view is fine):
    sum of bits(T[i][j]) * (2*(i*m + j) + 1) mod 2^64.  Sensitive to every bit of every cell
    (the weight is odd), cheap enough for 4.3 GB tables on both sides of the comparison."""
    n, m = body.shape
    acc = np.uint64(0)
    j2 = (np.arange(m, dtype=np.uint64) << np.uint64(1)) + np.uint64(1)
    with np.errstate(over="ignore"):
        for i0 in range(0, n, 256):
            blk = np.ascontiguousarray(body[i0:i0 + 256]).view(np.uint64)
            base = (np.arange(i0, i0 + blk.shape[0], dtype=np.uint64) * np.uint64(2 * m))[:, None]
            acc = acc + (blk * (base + j2[None, :])).sum(dtype=np.uint64)
    return int(acc)


def body_checksum_torch(body, m_total=None, col0: int = 0) -> int:
    """Same checksum for a device tensor view [n, m_loc] (fp64, any row stride); int64 wraps mod 2^64.
    A column shard passes the width of the whole table (m_total) and its first column (col0): the checksums of the
    shards then ADD UP (mod 2^64) to the checksum of the whole body."""
    import torch
    n, m = body.shape
    mt = int(m if m_total is None else m_total)
    dev = body.device
    j2 = (torch.arange(m, dtype=torch.int64, device=dev) + int(col0)) * 2 + 1
    acc = torch.zeros((), dtype=torch.int64, device=dev)
    for i0 in range(0, n, 1024):
        blk = body[i0:i0 + 1024].contiguous().view(torch.int64)
        base = (torch.arange(i0, i0 + blk.shape[0], dtype=torch.int64, device=dev) * (2 * mt))[:, None]
        acc = acc + (blk * (base + j2[None, :])).sum()
    return int(acc.item()) & 0xFFFFFFFFFFFFFFFF
