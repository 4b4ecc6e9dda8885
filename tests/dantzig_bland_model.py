"""An independent pure-Python statement of Dantzig's rule with Bland's rule on degenerate pivots and a ratio-tested
phase 1 (SPX_RULE_DANTZIG_BLAND, include/spx_b200.h) — test infrastructure only.  Python floats are IEEE binary64 with
every quotient rounded on its own, as in the kernels and in tests/dantzig_bland_oracle.c, which it is checked against.

t is the first row with b < 0.  Phase 1 (t exists) enters among the j with T[t][j] > 0, phase 2 among the j with
f_j < 0.  Dantzig's column has the largest T[t][j] or -f_j (lowest j on ties), Bland's the lowest header label.  The
leaving row of a column is the least (ratio, not target, row label, i) over row t and the rows with T[i][c] < 0 and
b_i not < 0; NaN ratios come after every number.  Bland's column replaces Dantzig's when Dantzig's step is +-0.
The pivot and the label swap are the reference's (devex_model.pivot).
"""
import math

from devex_model import pivot

PIVOT, OPTIMAL, INCORRECT, NOCONV, CAP = 1, 0, -1, -2, -3
ZERO = (0, 0.0)


def ratio_key(v):
    """numbers by value (-0.0 == 0.0 in Python), every NaN after every number and equal to every NaN"""
    return (1, 0.0) if math.isnan(v) else (0, v)


def leave(rows, m, c, t, cl):
    """the least (ratio key, not target, label, i) of column c, None when no row is a candidate"""
    best = None
    for i, row in enumerate(rows):
        a, b = row[c], row[m]
        if i == t:
            key = (ratio_key((0.0 - b) / a), 0, 0, i)
        elif a < 0 and not b < 0:
            key = (ratio_key(b / (0.0 - a)), 1, cl[i], i)
        else:
            continue
        if best is None or key < best:
            best = key
    return best


def pick(rows, f, rl, cl):
    """(status, r, c) of one pick: rows are the n body rows [a_1..a_m, b], f the f row, rl / cl the labels"""
    n, m = len(rows), len(f)
    t = next((i for i in range(n) if rows[i][m] < 0), None)
    if t is not None:
        cand = [j for j in range(m) if rows[t][j] > 0]
        score = [rows[t][j] for j in range(m)]
    else:
        cand = [j for j in range(m) if f[j] < 0]
        score = [-v for v in f]
    if not cand:
        return (INCORRECT if t is not None else OPTIMAL), -1, -1
    c = min(cand, key=lambda j: (-score[j], j))
    best = leave(rows, m, c, t, cl)
    if best is not None and best[0] == ZERO:
        c = min(cand, key=lambda j: (rl[j], j))
        best = leave(rows, m, c, t, cl)
    if best is None:
        return NOCONV, -1, -1
    return PIVOT, best[3], c


def solve(T, n, m, max_pivots, rowlab=None, collab=None):
    """A solve of the reference-flat table T (a sequence of floats) under the rule.
    Returns (status, trace [(r, c)], final flat table [floats], rowlab, collab)."""
    T = [float(v) for v in T]
    rows = [T[i * (m + 1): (i + 1) * (m + 1)] for i in range(n)]
    f = T[n * (m + 1):]
    rl = list(range(m)) if rowlab is None else [int(v) for v in rowlab]
    cl = list(range(m, m + n)) if collab is None else [int(v) for v in collab]
    trace = []
    while True:
        st, r, c = pick(rows, f, rl, cl)
        if st != PIVOT:
            break
        if len(trace) >= max_pivots:
            st = CAP
            break
        trace.append((r, c))
        rows, f = pivot(rows, f, r, c)
        rl[c], cl[r] = cl[r], rl[c]
    return st, trace, [v for row in rows for v in row] + f, rl, cl
