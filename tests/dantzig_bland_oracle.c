/* dantzig_bland_oracle.c — the sequential statement of Dantzig's rule with Bland's rule on degenerate pivots and a
 * ratio-tested phase 1 (SPX_RULE_DANTZIG_BLAND, include/spx_b200.h), test infrastructure only.  It is linked with
 * oracle/spx_oracle.c and uses that file's pivot (orc_update) and extraction unchanged: only the choice of (r, c) is
 * new here.  Compiled with -ffp-contract=off: every quotient is one correctly rounded division, as in the kernels.
 *
 * The table is the dictionary x_B = b + T x_N, f = f0 + sum d_j x_N_j.  Per pick:
 *   t        : the lowest row with b < 0, else none (phase 2)
 *   phase 1  : candidates j with T[t][j] > 0 (none: INCORRECT), score T[t][j]
 *   phase 2  : candidates j with f[j] < 0 (none: OPTIMAL), score -f[j]
 *   c_D      : the largest score, lowest j on ties;  c_B: the lowest header label rowlab[j], lowest j on ties
 *   leave(c) : the least (ratio, not_target, label, i) over the target row t (ratio (0 - b_t) / T[t][c], 0, 0) and
 *              the rows i != t with T[i][c] < 0 and !(b_i < 0) (ratio b_i / (0 - T[i][c]), 1, collab[i]); ratios
 *              compare as numbers, -0 = +0, every NaN after every number and equal to every NaN; no row: NOCONV
 *   pick     : (leave(c_D), c_D), unless that ratio is +-0: then (leave(c_B), c_B) */
#include <stdint.h>
#include <stddef.h>
#include <string.h>

#define ORC_PIVOT      1
#define ORC_OPTIMAL    0
#define ORC_INCORRECT -1
#define ORC_NOCONV    -2
#define ORC_CAP       -3

void orc_update(const double *T, double *N, int n, int m, int r, int c);

static inline size_t row_off(int i, int m) { return (size_t)i * (size_t)(m + 1); }

/* -1, 0, 1 as ratio a comes before, ties with, or comes after ratio b */
static int cmp_ratio(double a, double b)
{
    const int na = a != a, nb = b != b;
    if (na || nb) return na - nb;
    return (a > b) - (a < b);
}

/* the leaving row of column c (t: the target row or -1), -1 when no row is a candidate; *ratio = its ratio */
static int leave(const double *T, int n, int m, int c, int t, const int32_t *collab, double *ratio)
{
    int best = -1, bnt = 0;
    int32_t blab = 0;
    double br = 0.0;
    for (int i = 0; i < n; ++i) {
        const double a = T[row_off(i, m) + c], b = T[row_off(i, m) + m];
        double q;
        int nt;
        int32_t lab;
        if (i == t) { q = (0.0 - b) / a; nt = 0; lab = 0; }
        else if (a < 0 && !(b < 0)) { q = b / (0.0 - a); nt = 1; lab = collab[i]; }
        else continue;
        int k = best < 0 ? -1 : cmp_ratio(q, br);
        if (k == 0) k = nt - bnt;
        if (k == 0) k = (lab > blab) - (lab < blab);
        if (k < 0) { best = i; br = q; bnt = nt; blab = lab; }     /* rows ascend: a full tie keeps the lower i */
    }
    *ratio = br;
    return best;
}

int orc_pick_db(const double *T, int n, int m, const int32_t *rowlab, const int32_t *collab, int *r_out, int *c_out)
{
    int t = -1;
    for (int i = 0; i < n; ++i)
        if (T[row_off(i, m) + m] < 0) { t = i; break; }
    const double *e = T + row_off(t >= 0 ? t : n, m);
    int cd = -1, cb = -1;
    double sd = 0.0;
    for (int j = 0; j < m; ++j) {
        const double v = e[j];
        if (!(t >= 0 ? v > 0 : v < 0)) continue;
        const double s = t >= 0 ? v : -v;
        if (cd < 0 || s > sd) { cd = j; sd = s; }
        if (cb < 0 || rowlab[j] < rowlab[cb]) cb = j;
    }
    if (cd < 0) return t >= 0 ? ORC_INCORRECT : ORC_OPTIMAL;
    double q;
    int c = cd, r = leave(T, n, m, cd, t, collab, &q);
    if (r < 0) return ORC_NOCONV;                          /* c_D is a ray (phase 2 only) */
    if (q == 0) {                                          /* a degenerate step */
        c = cb;
        r = leave(T, n, m, cb, t, collab, &q);
        if (r < 0) return ORC_NOCONV;
    }
    *r_out = r; *c_out = c;
    return ORC_PIVOT;
}

/* orc_solve_rule of oracle/spx_oracle.c with this pick; rowlab / collab are the labels to start from (a fresh solve
 * passes orc_init_labels') and are updated in place */
int orc_solve_db(double *T, double *scratch, int n, int m, int64_t max_pivots, int32_t *trace, double *snaps,
                 int32_t *rowlab, int32_t *collab, int64_t *npiv_out)
{
    const size_t cells = (size_t)n * (size_t)(m + 1) + (size_t)m;
    double *cur = T, *nxt = scratch;
    int64_t k = 0;
    int status;
    if (snaps) memcpy(snaps, cur, cells * sizeof(double));
    for (;;) {
        int r = 0, c = 0;
        status = orc_pick_db(cur, n, m, rowlab, collab, &r, &c);
        if (status != ORC_PIVOT) break;
        if (k >= max_pivots) { status = ORC_CAP; break; }
        if (trace) { trace[2 * k] = r; trace[2 * k + 1] = c; }
        orc_update(cur, nxt, n, m, r, c);
        { int32_t t = rowlab[c]; rowlab[c] = collab[r]; collab[r] = t; }
        double *t = cur; cur = nxt; nxt = t;
        ++k;
        if (snaps) memcpy(snaps + (size_t)k * cells, cur, cells * sizeof(double));
    }
    if (cur != T) memcpy(T, cur, cells * sizeof(double));
    *npiv_out = k;
    return status;
}
