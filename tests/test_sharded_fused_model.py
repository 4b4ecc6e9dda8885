"""CPU model of the column-sharded FUSED loop (csrc/spx_fused.cu: shard_price_kernel + update_lazy_kernel),
checked bit for bit against the oracle.  It restates, in numpy and rank by rank, WHAT every rank computes in
a pass — not the CUDA code — so that the algorithm the kernels implement is pinned on the inputs the hardware
tests could not cover in round 1 (entering columns owned by the LAST ranks, phase-1 pivots, degenerate ties,
early endings, ranks without columns, look-ahead with up to 2F-1 pending levels):

  per level i of a pass, on every rank            (reference rule: simplex.py:70-141, arithmetic :143-177)
    A  running b (replicated), running local f-row shard, local shard of ROW_{i-1} by gather + replay
    .  r1 = first b < 0;  local candidate = first positive cell of virtual row r1 (phase 1) or the first
       negative local f cell;  key = global column index
    B  the rank's candidate COLUMN of the virtual table (gather + replay), stored speculatively
    X  exchange: lexicographic-minimum key wins -> (global column, owner); everyone reads the owner's column
    R  ratio test on that column against the running b (replicated, identical on every rank)
  after the levels: every rank applies the pass's levels to its own columns in one sweep.
  Look-ahead: the levels of pass q+1 are priced from the table BEFORE pass q's sweep, replaying pass q's levels first.

Every cell goes through the reference's separately rounded operations, so trace, labels, status and all
table bits must equal the pivot-at-a-time oracle's.
"""
import numpy as np
import pytest

import oracle
from simplex_method_solver_b200 import workloads as W
from util import bits, make_lp, owners_of

NONE = 1 << 30


def apply_level(v, t, j, lvl, rowval, colval):
    """cell(s) (t, j) after one more pending pivot.  lvl = (r, c_local or -1, p); rowval = ROW_l[j], colval = COL_l[t]."""
    r, c, p = lvl
    v, t, j, rowval, colval = np.broadcast_arrays(np.asarray(v, dtype=np.float64), t, j, rowval, colval)
    with np.errstate(all="ignore"):
        general = (v * p - rowval * colval) / p
        out = np.where((t == r) & (j == c), np.float64(1.0) / p,
                       np.where(t == r, (-v) / p, np.where(j == c, colval / p, general)))
    return out.astype(np.float64)


def ratio_row(col, b, n):
    """leaving row by the reference's ratio rule (simplex.py:107-136), through the oracle's own pick on the
    one-column table [col | b] with a negative objective cell: (row or -1 for 'does not converge')"""
    T = np.empty(n * 2 + 1)
    T[0:2 * n:2] = col[:n]
    T[1:2 * n:2] = b
    T[2 * n] = -1.0
    st, r, c, p = oracle.pick(T, n, 1)
    return r if st == oracle.PIVOT else -1


class Rank:
    def __init__(self, body, frow, col0):
        self.A = body.copy()              # stored table: [n, m_loc] local columns
        self.f = frow.copy()              # stored f row shard
        self.col0, self.m = col0, body.shape[1]
        self.frow = None                  # running f-row shard while pricing
        self.ROW = []                     # ROW planes of the levels this rank still has pending (local shards)


def run_model(rows, c, splits, F, cap, lookahead):
    n, m = rows.shape[0], rows.shape[1] - 1
    ranks = [Rank(rows[:, a:z], c[a:z], a) for a, z in splits]
    b_stored = rows[:, m].copy()
    rowlab, collab = oracle.init_labels(n, m)
    rowlab, collab = list(rowlab), list(collab)
    trace, status = [], oracle.PIVOT
    pending = []                          # look-ahead: levels priced but not yet swept: dicts r, c, p, COL, owner

    def local(lvl, rk):
        cl = lvl["c"] - rk.col0
        return (lvl["r"], cl if 0 <= cl < rk.m else -1, lvl["p"])

    def sweep(levels, row_planes_per_rank):
        """update_lazy_kernel: every rank applies `levels` to its stored columns (and f row shard)"""
        for rk, planes in zip(ranks, row_planes_per_rank):
            if rk.m == 0:
                continue
            T = np.vstack([rk.A, rk.f[None, :]])
            tt, jj = np.meshgrid(np.arange(n + 1), np.arange(rk.m), indexing="ij")
            for lvl, ROW in zip(levels, planes):
                T = apply_level(T, tt, jj, local(lvl, rk), ROW[None, :], lvl["COL"][:, None])
            rk.A, rk.f = T[:n], T[n]

    while status == oracle.PIVOT:
        # ------------------------------------------------ shard_price_kernel, one pass
        prev = pending                                        # np levels the stored tables do not contain yet
        prev_rows = [list(rk.ROW) for rk in ranks]
        levels = []
        for rk in ranks:
            rk.ROW = []
            if not prev:
                rk.frow = rk.f.copy()                         # else: the previous pricing left it at this table
        bv = b_stored.copy()
        for i in range(F + 1):
            allv = prev + levels
            if i > 0:
                L = levels[i - 1]
                br, COLL = bv[L["r"]], L["COL"]
                with np.errstate(all="ignore"):
                    nb = (bv * L["p"] - br * COLL[:n]) / L["p"]
                    nb[L["r"]] = (-bv[L["r"]]) / L["p"]
                bv = nb
                for k, rk in enumerate(ranks):                # ROW_{i-1} and the running f row, local shard
                    jj = np.arange(rk.m)
                    rv = rk.A[L["r"]].copy()
                    for l, lv in enumerate(allv[:-1]):
                        rp = (prev_rows[k] + rk.ROW)[l]
                        rv = apply_level(rv, L["r"], jj, local(lv, rk), rp, lv["COL"][L["r"]])
                    rk.ROW.append(rv)
                    cl = local(L, rk)[1]
                    with np.errstate(all="ignore"):
                        nf = (rk.frow * L["p"] - rv * COLL[n]) / L["p"]
                        if cl >= 0:
                            nf[cl] = COLL[n] / L["p"]
                    rk.frow = nf
            if i == F:
                break
            neg = np.flatnonzero(bv < 0.0)
            r1 = int(neg[0]) if len(neg) else -1
            keys, cols = [], []
            for k, rk in enumerate(ranks):
                jj = np.arange(rk.m)
                planes = prev_rows[k] + rk.ROW
                if r1 >= 0:                                   # first positive cell of the virtual row r1
                    v = rk.A[r1].copy()
                    for l, lv in enumerate(allv):
                        v = apply_level(v, r1, jj, local(lv, rk), planes[l], lv["COL"][r1])
                    hit = np.flatnonzero(v > 0.0)
                else:
                    hit = np.flatnonzero(rk.frow < 0.0)
                cloc = int(hit[0]) if len(hit) else NONE
                keys.append(NONE if cloc == NONE else rk.col0 + cloc)
                if cloc == NONE:
                    cols.append(None)
                    continue
                tt = np.arange(n + 1)
                w = np.concatenate([rk.A[:, cloc], rk.f[cloc: cloc + 1]])
                for l, lv in enumerate(allv):
                    w = apply_level(w, tt, cloc, local(lv, rk), planes[l][cloc], lv["COL"])
                cols.append(w)
            cglob = min(keys)
            if cglob == NONE:
                status = oracle.INCORRECT if r1 >= 0 else oracle.OPTIMAL
                break
            owner = keys.index(cglob)
            COL = cols[owner]
            r = r1 if r1 >= 0 else ratio_row(COL, bv, n)
            if r < 0:
                status = oracle.NOCONV
                break
            if len(trace) >= cap:
                status = oracle.CAP
                break
            levels.append({"r": r, "c": cglob, "p": COL[r], "COL": COL, "owner": owner})
            rowlab[cglob], collab[r] = collab[r], rowlab[cglob]
            trace.append((r, cglob))
        b_next = bv
        # ------------------------------------------------ the sweeps
        if lookahead:
            if prev:
                sweep(prev, prev_rows)                        # U_q runs while P_{q+1} (above) priced from its input
            pending = levels
            if status != oracle.PIVOT and levels:
                sweep(levels, [rk.ROW for rk in ranks])
        else:
            if levels:
                sweep(levels, [rk.ROW for rk in ranks])
            for rk in ranks:
                rk.ROW = []
        b_stored = b_next
    body = np.zeros((n + 1, m))
    for rk in ranks:
        body[:n, rk.col0: rk.col0 + rk.m] = rk.A
        body[n, rk.col0: rk.col0 + rk.m] = rk.f
    return status, trace, body, b_stored, rowlab, collab


def splits_of(m, widths):
    out, a = [], 0
    for w in widths:
        z = min(m, a + w)
        out.append((a, z))
        a = z
    assert a == m
    return out


CASES = [
    # n, m, seed, kind, widths of the ranks' column blocks, F, cap
    (6, 10, 1, "dense", [4, 4, 2], 3, 40),
    (9, 40, 7, "dense", [40, 0], 5, 60),                      # rank 1 owns nothing
    (12, 60, 3, "late", [32, 28], 5, 60),                     # the entering column lives on the last rank
    (20, 160, 3, "late", [50, 50, 30, 30], 4, 70),            # ... and moves between all four ranks
    (30, 150, 5, "late", [100, 50], 8, 90),
    (40, 400, 1, "late", [128, 128, 144], 8, 90),             # 64 pivots, 22 owner changes
    (48, 600, 2, "late", [200, 0, 200, 200], 5, 100),         # an empty rank in the middle
    (12, 70, 7, "smallint", [8, 30, 32], 5, 60),              # phase-1 pivots, ties, 'does not converge'
    (7, 33, 8, "smallint", [11, 11, 11], 3, 40),
    (20, 44, 9, "smallint", [4, 20, 20], 8, 80),              # 80 pivots (cap), 33 owner changes
    (14, 96, 13, "smallint", [3, 3, 90], 2, 60),
    (5, 30, 12, "smallint", [10, 0, 20], 2, 7),
]


@pytest.mark.parametrize("lookahead", [False, True])
@pytest.mark.parametrize("n,m,seed,kind,widths,F,cap", CASES)
def test_sharded_fused_model_equals_oracle(n, m, seed, kind, widths, F, cap, lookahead):
    rows, c = make_lp(n, m, seed, kind)
    o = oracle.solve(rows, c, max_pivots=cap)
    status, trace, body, b, rowlab, collab = run_model(rows, c, splits_of(m, widths), F, cap, lookahead)
    assert (status, len(trace)) == (o.status, o.npiv)
    assert [list(t) for t in trace] == o.trace.tolist()
    assert list(rowlab) == o.rowlab.tolist() and list(collab) == o.collab.tolist()
    ot = o.table[: n * (m + 1)].reshape(n, m + 1)
    ob = np.vstack([ot[:, :m], o.table[n * (m + 1):][None, :]])
    same = (bits(body) == bits(ob)) | (np.isnan(body) & np.isnan(ob))
    assert same.all(), np.argwhere(~same)[:5]
    sameb = (bits(b) == bits(ot[:, m].copy())) | (np.isnan(b) & np.isnan(ot[:, m]))
    assert sameb.all()


def test_cases_cover_what_they_claim():
    """the cases really have entering columns on every rank, owner changes, phase-1 pivots and all endings"""
    owners, endings, phase1, switches = set(), set(), 0, 0
    for n, m, seed, kind, widths, F, cap in CASES:
        rows, c = make_lp(n, m, seed, kind)
        o = oracle.solve(rows, c, max_pivots=cap)
        endings.add(o.status)
        own = owners_of(o.trace.tolist(), [(a, z - a) for a, z in splits_of(m, widths)])
        owners.update((kind, g) for g in own)
        switches += sum(a != b for a, b in zip(own, own[1:]))
        T = np.concatenate([rows.reshape(-1), c])
        for r, cc in o.trace.tolist():
            if (T[m: n * (m + 1): m + 1] < 0).any():
                phase1 += 1
            T = oracle.update(T, n, m, r, cc)
    assert {g for k, g in owners if k == "late"} >= {0, 1, 2, 3}
    assert {g for k, g in owners if k == "smallint"} >= {0, 1, 2}
    assert switches > 80 and phase1 > 10, (switches, phase1)
    assert endings >= {oracle.OPTIMAL, oracle.NOCONV, oracle.CAP}, endings
