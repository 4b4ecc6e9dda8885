/*
 * certificate_oracle.c — sequential CPU statement of the certificate report (spx_certificate_*, include/spx_b200.h).
 *
 * TEST INFRASTRUCTURE ONLY: tests/test_certificate.py and __graft_entry__.smoke() compile it into a temporary
 * directory and check the device kernels against it bit for bit.  It sits beside the tests rather than in oracle/,
 * whose pinned restatement of the reference it does not change.
 *
 * The final table T is reference flat (n rows of [T[i][0..m-1], b_i], then the f row d_0..d_{m-1}) with int32 labels
 * (x_k -> k, y_k -> m + k; rowlab over the columns, collab over the rows).  It is the dictionary x_B = b + T x_N,
 * f = f0 + sum_j d_j x_N of "minimise c.x subject to b + A x >= 0, x >= 0".
 *
 *   Farkas row:  the lowest i with b_i finite and < 0 and every T[i][j] (j < m) finite and <= 0, else -1.
 *                farkas [n] = +0.0; farkas[L-m] = 1.0 for L = collab[r] a y label; then for j ascending,
 *                farkas[H-m] = 0.0 - T[r][j] for H = rowlab[j] a y label.  bound = b_r.
 *   Ray column:  only when every b_i is finite and >= 0: the lowest j with d_j finite and < 0 and every T[i][j]
 *                (i < n) finite and >= 0, else -1.
 *                ray [m] = +0.0; ray[H] = 1.0 for H = rowlab[c] an x label; then for i ascending,
 *                ray[L] = T[i][c] + 0.0 for L = collab[i] an x label.  slope = d_c.
 * Without a certificate its vector and its bound (slope) are NaN.  A label outside its range is skipped.
 * Build with -ffp-contract=off and without -ffast-math.
 */
#include <math.h>
#include <stdint.h>
#include <stddef.h>


void orc_certificate(const double *T, int n, int m, const int32_t *rowlab, const int32_t *collab,
                     int32_t *row, double *farkas, double *bound, int32_t *col, double *ray, double *slope)
{
    const size_t w = (size_t)m + 1;
    const double *f = T + (size_t)n * w;
    int r = -1;
    for (int i = 0; i < n && r < 0; ++i) {
        const double bi = T[i * w + m];
        if (!(isfinite(bi) && bi < 0)) continue;
        int ok = 1;
        for (int j = 0; j < m; ++j)
            if (!(isfinite(T[i * w + j]) && T[i * w + j] <= 0)) { ok = 0; break; }
        if (ok) r = i;
    }
    *row = r;
    if (r < 0) {
        for (int k = 0; k < n; ++k) farkas[k] = NAN;
        *bound = NAN;
    } else {
        for (int k = 0; k < n; ++k) farkas[k] = 0.0;
        const int32_t L = collab[r];
        if (L >= m && L < m + n) farkas[L - m] = 1.0;
        for (int j = 0; j < m; ++j) {
            const int32_t H = rowlab[j];
            if (H >= m && H < m + n) farkas[H - m] = 0.0 - T[r * w + j];
        }
        *bound = T[r * w + m];
    }

    int feasible = 1;
    for (int i = 0; i < n; ++i) {
        const double bi = T[i * w + m];
        if (!(isfinite(bi) && bi >= 0)) feasible = 0;
    }
    int c = -1;
    for (int j = 0; feasible && j < m && c < 0; ++j) {
        if (!(isfinite(f[j]) && f[j] < 0)) continue;
        int ok = 1;
        for (int i = 0; i < n; ++i)
            if (!(isfinite(T[i * w + j]) && T[i * w + j] >= 0)) { ok = 0; break; }
        if (ok) c = j;
    }
    *col = c;
    if (c < 0) {
        for (int k = 0; k < m; ++k) ray[k] = NAN;
        *slope = NAN;
    } else {
        for (int k = 0; k < m; ++k) ray[k] = 0.0;
        const int32_t H = rowlab[c];
        if (H >= 0 && H < m) ray[H] = 1.0;
        for (int i = 0; i < n; ++i) {
            const int32_t L = collab[i];
            if (L >= 0 && L < m) ray[L] = T[i * w + c] + 0.0;
        }
        *slope = f[c];
    }
}
