/*
 * sensitivity_oracle.c — sequential CPU statement of the sensitivity report (spx_sensitivity_*, include/spx_b200.h).
 *
 * TEST INFRASTRUCTURE ONLY: tests/test_sensitivity.py and __graft_entry__.smoke() compile it into a temporary
 * directory and check the device kernels against it bit for bit.  It sits beside the tests rather than in oracle/,
 * whose pinned restatement of the reference it does not change.
 *
 * The final table T is reference flat (n rows of [T[i][0..m-1], b_i], then the f row d_0..d_{m-1}) with int32 labels
 * (x_k -> k, y_k -> m + k; rowlab over the columns, collab over the rows).  It is a dictionary: x_B = b + T x_N and
 * f = f0 + sum_j d_j x_N.  Per constraint k: dual, slack [n], rhs_range [n][2]; per variable k: redcost [m],
 * cost_range [m][2]:
 *   y_k nonbasic in column j: -d_j, 0, (min_{i: T[i][j] < 0} b_i / (-T[i][j]), min_{i: T[i][j] > 0} b_i / T[i][j])
 *   y_k basic in row i:       0, b_i, (b_i, +inf)
 *   x_k nonbasic in column j: d_j, (d_j, +inf)
 *   x_k basic in row i:       0, (min_{j: T[i][j] > 0} d_j / T[i][j], min_{j: T[i][j] < 0} d_j / (-T[i][j]))
 * A minimum over an empty set is +inf, a NaN quotient never wins, every zero is +0.0, and when optimal == 0 every
 * output is NaN.  Build with -ffp-contract=off and without -ffast-math: each quotient is one IEEE division.
 */
#include <math.h>
#include <stdint.h>
#include <stddef.h>

static double pos0(double v) { return v == 0.0 ? 0.0 : v; }

void orc_sensitivity(const double *T, int n, int m, const int32_t *rowlab, const int32_t *collab, int optimal,
                     double *dual, double *slack, double *redcost, double *rhs_range, double *cost_range)
{
    const size_t w = (size_t)m + 1;
    const double *f = T + (size_t)n * w;
    if (!optimal) {
        for (int k = 0; k < n; ++k) dual[k] = slack[k] = rhs_range[2 * k] = rhs_range[2 * k + 1] = NAN;
        for (int k = 0; k < m; ++k) redcost[k] = cost_range[2 * k] = cost_range[2 * k + 1] = NAN;
        return;
    }
    for (int i = 0; i < n; ++i) {
        const int32_t lab = collab[i];
        const double bi = pos0(T[i * w + m]);
        if (lab >= m) {
            const int k = lab - m;
            dual[k] = 0.0; slack[k] = bi;
            rhs_range[2 * k] = bi; rhs_range[2 * k + 1] = INFINITY;
        } else {
            double dec = INFINITY, inc = INFINITY;
            for (int j = 0; j < m; ++j) {
                const double t = T[i * w + j];
                if (t > 0) { const double q = f[j] / t; if (q < dec) dec = q; }
                else if (t < 0) { const double q = f[j] / (-t); if (q < inc) inc = q; }
            }
            redcost[lab] = 0.0;
            cost_range[2 * lab] = pos0(dec); cost_range[2 * lab + 1] = pos0(inc);
        }
    }
    for (int j = 0; j < m; ++j) {
        const int32_t lab = rowlab[j];
        const double d = f[j];
        if (lab >= m) {
            const int k = lab - m;
            double dec = INFINITY, inc = INFINITY;
            for (int i = 0; i < n; ++i) {
                const double t = T[i * w + j], bi = T[i * w + m];
                if (t < 0) { const double q = bi / (-t); if (q < dec) dec = q; }
                else if (t > 0) { const double q = bi / t; if (q < inc) inc = q; }
            }
            dual[k] = pos0(-d); slack[k] = 0.0;
            rhs_range[2 * k] = pos0(dec); rhs_range[2 * k + 1] = pos0(inc);
        } else {
            redcost[lab] = pos0(d);
            cost_range[2 * lab] = pos0(d); cost_range[2 * lab + 1] = INFINITY;
        }
    }
}
