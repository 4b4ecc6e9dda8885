"""An independent pure-Python statement of the devex entering rule (SPX_RULE_DEVEX, include/spx_b200.h) on top of
the reference's loop — test infrastructure only.  Python floats are IEEE binary64 with every product, difference
and quotient rounded on its own, as in the kernels and in tests/devex_oracle.c, which it is checked against.

The reference's phase 1 (simplex.py:72-91), ratio scan (:107-136) and out-of-place pivot (:149-177) with labels
(:152); the entering column of phase 2 is the largest (f_j * f_j) / w_j over f_j < 0 (NaN below every number, the
lowest j on ties), and after every pivot (r, c) with u = row r of the new table and t_j = (u_j * u_j) * w_c (the old
w_c): w_j = max(w_j, t_j) for j != c and w_c = max(1, t_c), where a NaN t never replaces a weight.
"""
import math

PIVOT, OPTIMAL, INCORRECT, NOCONV, CAP = 1, 0, -1, -2, -3


def pick(rows, f, w):
    """(status, r, c) of one pick: rows are the n body rows [a_1..a_m, b], f the f row, w the weights"""
    n, m = len(rows), len(f)
    for i in range(n):
        if rows[i][m] < 0:
            for j in range(m):
                if rows[i][j] > 0:
                    return PIVOT, i, j
            return INCORRECT, -1, -1
    col, best = -1, 0.0
    for j in range(m):
        if f[j] < 0:
            s = (f[j] * f[j]) / w[j]
            if col < 0 or (not math.isnan(s) and (math.isnan(best) or s > best)):
                col, best = j, s
    if col < 0:
        return OPTIMAL, -1, -1
    row, first, min_val = -1, True, 1.0
    for i in range(n):
        a = rows[i][col]
        if a == 0:
            continue
        val = rows[i][m] / a
        if first:
            min_val, row, first = val, i, False
        elif val == 0 and min_val > 0:
            min_val, row = val, i
        elif val < 0 and 0 <= min_val:
            min_val, row = val, i
        elif min_val <= val < 0:
            min_val, row = val, i
    if first or min_val > 0:
        return NOCONV, -1, -1
    return PIVOT, row, col


def pivot(rows, f, r, c):
    """the reference's out-of-place pivot: new (rows, f)"""
    p, prow = rows[r][c], rows[r]
    new = []
    for i, src in enumerate(rows + [f]):
        if i == r:
            dst = [-v / p for v in src]
            dst[c] = 1.0 / p
        else:
            ci = src[c]
            dst = [(v * p - prow[j] * ci) / p for j, v in enumerate(src)]
            dst[c] = ci / p
        new.append(dst)
    return new[:-1], new[-1]


def update_weights(w, u, c):
    """the weights after a pivot in column c whose new pivot row is u"""
    wc = w[c]
    out = []
    for j, wj in enumerate(w):
        t = (u[j] * u[j]) * wc
        out.append((t if t > 1.0 else 1.0) if j == c else (t if t > wj else wj))
    return out


def solve(T, n, m, max_pivots, rowlab=None, collab=None):
    """A devex solve of the reference-flat table T (a sequence of floats) from unit weights.
    Returns (status, trace [(r, c)], final flat table [floats], rowlab, collab)."""
    T = [float(v) for v in T]
    rows = [T[i * (m + 1): (i + 1) * (m + 1)] for i in range(n)]
    f = T[n * (m + 1):]
    rl = list(range(m)) if rowlab is None else [int(v) for v in rowlab]
    cl = list(range(m, m + n)) if collab is None else [int(v) for v in collab]
    w = [1.0] * m
    trace = []
    while True:
        st, r, c = pick(rows, f, w)
        if st != PIVOT:
            break
        if len(trace) >= max_pivots:
            st = CAP
            break
        trace.append((r, c))
        rows, f = pivot(rows, f, r, c)
        w = update_weights(w, rows[r], c)
        rl[c], cl[r] = cl[r], rl[c]
    return st, trace, [v for row in rows for v in row] + f, rl, cl
