/* devex_oracle.c — the sequential statement of the devex entering rule (SPX_RULE_DEVEX, include/spx_b200.h), test
 * infrastructure only.  It is linked with oracle/spx_oracle.c and uses that file's pivot (orc_update), labels
 * (orc_init_labels) and extraction unchanged: only the entering column of phase 2 and the weights are new here.
 * Phase 1 (simplex.py:72-91) and the ratio scan (:107-136) are restated as in orc_pick_rule.
 * Compiled with -ffp-contract=off: every product and quotient is rounded on its own, as in the kernels.
 *
 * Weights w[0..m), one per column of the f row, all 1 at the start of every solve and resume.
 *   entering : among j with f[j] < 0 (NaN never), the largest score (f[j]*f[j]) / w[j], NaN below every number,
 *              the lowest j on ties
 *   update   : after EVERY pivot (r, c), phase-1 pivots included, with u = row r of the new table and
 *              t_j = (u_j*u_j) * w_old[c]:  w[j] = t_j > w[j] ? t_j : w[j] (j != c),  w[c] = t_c > 1 ? t_c : 1 */
#include <stdint.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>

#define ORC_PIVOT      1
#define ORC_OPTIMAL    0
#define ORC_INCORRECT -1
#define ORC_NOCONV    -2
#define ORC_CAP       -3

void orc_update(const double *T, double *N, int n, int m, int r, int c);

static inline size_t row_off(int i, int m) { return (size_t)i * (size_t)(m + 1); }

/* is score a better than score b (NaN below every number; ties are not better) */
static int better(double a, double b)
{
    if (a != a) return 0;
    if (b != b) return 1;
    return a > b;
}

int orc_pick_devex(const double *T, int n, int m, const double *w, int *r_out, int *c_out, double *e_out)
{
    int target_row = -1, target_col = -1;
    for (int i = 0; i < n; ++i)
        if (T[row_off(i, m) + m] < 0) { target_row = i; break; }
    if (target_row >= 0) {
        const double *row = T + row_off(target_row, m);
        for (int j = 0; j < m; ++j)
            if (row[j] > 0) { target_col = j; break; }
        if (target_col < 0) return ORC_INCORRECT;
        *r_out = target_row; *c_out = target_col; *e_out = row[target_col];
        return ORC_PIVOT;
    }
    const double *f = T + row_off(n, m);
    double best = 0.0;
    for (int j = 0; j < m; ++j) {
        if (!(f[j] < 0)) continue;
        const double fj2 = f[j] * f[j];
        const double s = fj2 / w[j];
        if (target_col < 0 || better(s, best)) { best = s; target_col = j; }
    }
    if (target_col < 0) return ORC_OPTIMAL;

    int first_try = 1;
    double min_val = 1;
    for (int i = 0; i < n; ++i) {
        double a = T[row_off(i, m) + target_col];
        if (a == 0) continue;
        double val = T[row_off(i, m) + m] / a;
        if (first_try) { min_val = val; target_row = i; first_try = 0; continue; }
        if (val == 0 && min_val > 0) { min_val = val; target_row = i; continue; }
        if (val < 0 && 0 <= min_val) { min_val = val; target_row = i; continue; }
        if (min_val <= val && val < 0) { min_val = val; target_row = i; continue; }
    }
    if (first_try || min_val > 0) return ORC_NOCONV;
    *r_out = target_row; *c_out = target_col;
    *e_out = T[row_off(target_row, m) + target_col];
    return ORC_PIVOT;
}

/* the weights after pivot (r, c); Tnew is the table that pivot produced */
void orc_devex_update(double *w, const double *Tnew, int n, int m, int r, int c)
{
    (void)n;
    const double *u = Tnew + row_off(r, m);
    const double wc = w[c];
    for (int j = 0; j < m; ++j) {
        const double u2 = u[j] * u[j];
        const double t = u2 * wc;
        if (j == c) w[j] = t > 1.0 ? t : 1.0;
        else w[j] = t > w[j] ? t : w[j];
    }
}

/* orc_solve_rule of oracle/spx_oracle.c with the devex pick; rowlab / collab are updated as given (a resume passes
 * the labels of its final table, a fresh solve orc_init_labels') */
int orc_solve_devex(double *T, double *scratch, int n, int m, int64_t max_pivots, int32_t *trace, double *snaps,
                    int32_t *rowlab, int32_t *collab, int64_t *npiv_out)
{
    const size_t cells = (size_t)n * (size_t)(m + 1) + (size_t)m;
    double *w = (double *)malloc((size_t)(m > 0 ? m : 1) * sizeof(double));
    for (int j = 0; j < m; ++j) w[j] = 1.0;
    double *cur = T, *nxt = scratch;
    int64_t k = 0;
    int status;
    if (snaps) memcpy(snaps, cur, cells * sizeof(double));
    for (;;) {
        int r = 0, c = 0; double e = 0;
        status = orc_pick_devex(cur, n, m, w, &r, &c, &e);
        if (status != ORC_PIVOT) break;
        if (k >= max_pivots) { status = ORC_CAP; break; }
        if (trace) { trace[2 * k] = r; trace[2 * k + 1] = c; }
        orc_update(cur, nxt, n, m, r, c);
        orc_devex_update(w, nxt, n, m, r, c);
        if (rowlab && collab) { int32_t t = rowlab[c]; rowlab[c] = collab[r]; collab[r] = t; }
        double *t = cur; cur = nxt; nxt = t;
        ++k;
        if (snaps) memcpy(snaps + (size_t)k * cells, cur, cells * sizeof(double));
    }
    if (cur != T) memcpy(T, cur, cells * sizeof(double));
    free(w);
    *npiv_out = k;
    return status;
}
