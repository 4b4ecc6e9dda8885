/* warm_oracle.c — the sequential statement of the change of final tables (spx_warm_change_batched / _ragged,
 * include/spx_b200.h), test infrastructure only.  Compiled with -ffp-contract=off: every product and sum is rounded
 * on its own, as in the kernel.
 *
 * One LP: T reference-flat (n rows of m+1 cells, then the f row of m cells), rowlab [m], collab [n] with codes
 * x_k -> k, y_k -> m + k; db [n] (or NULL), dc [m] (or NULL).  In place. */
#include <stdint.h>
#include <stddef.h>

void orc_warm_change(double *T, int n, int m, const int32_t *rowlab, const int32_t *collab, const double *db,
                     const double *dc)
{
    const size_t w1 = (size_t)m + 1;
    if (db) {
        for (int i = 0; i < n; ++i) {
            double v = T[i * w1 + m];
            const int L = collab[i];
            if (L >= m && L - m < n && db[L - m] != 0.0) v = v + db[L - m];
            for (int j = 0; j < m; ++j) {
                const int H = rowlab[j];
                if (H >= m && H - m < n) {
                    const double d = db[H - m];
                    if (d != 0.0) v = v - d * T[i * w1 + j];
                }
            }
            T[i * w1 + m] = v;
        }
    }
    if (dc) {
        double *f = T + (size_t)n * w1;
        for (int j = 0; j < m; ++j) {
            double v = f[j];
            const int H = rowlab[j];
            if (H >= 0 && H < m && dc[H] != 0.0) v = v + dc[H];
            for (int i = 0; i < n; ++i) {
                const int L = collab[i];
                if (L >= 0 && L < m) {
                    const double d = dc[L];
                    if (d != 0.0) v = v + d * T[i * w1 + j];
                }
            }
            f[j] = v;
        }
    }
}
