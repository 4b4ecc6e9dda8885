// spx_warm.cu — the change of final tables: new right-hand sides and costs applied to the dictionaries K4, K7 and K8
// leave, so that a resume (spx_warm_solve_*) re-optimises from them instead of from the first pivot.
//
// A final table is the dictionary  basic = b + T nonbasic,  f = const + sum_j d_j nonbasic_j  (recalculate_matrix,
// :143-177) of "minimise c.x subject to b + A x >= 0, x >= 0"; constraint k's slack is y_k, label codes x_k -> k,
// y_k -> m + k.  Moving b_k by db_k moves every basic variable by db_k times its column of y_k; moving c_k by dc_k
// moves every d_j by dc_k times row x_k.  Per LP, in this order (include/spx_b200.h states it too):
//   row i:     v = b_i;  v += db[collab[i] - m] if row i is y_k;  for j ascending with header y_k, db_k != 0:
//              v -= db_k * T[i][j];  b_i = v
//   column j:  v = d_j;  v += dc[rowlab[j]] if column j is x_k;  for i ascending with label x_k, dc_k != 0:
//              v += dc_k * T[i][j];  d_j = v
// Every product and sum is rounded on its own (__dmul_rn / __dadd_rn / __dsub_rn, never fused), a zero delta (-0.0
// included) is skipped, and a label outside its range is never used as an index.  The b update reads only body
// columns j < m and writes only column m; the f update reads only body rows and writes only the f row: both run in
// place, in one launch.
//
// Layout.  One grid over (tile, LP): blockIdx.x < tb is row tile blockIdx.x of the b update, the rest are column
// tiles of the f update; LPs stride over blockIdx.y.  A CTA walks the other dimension in chunks of WARM_THREADS,
// compacts the chunk's active columns (headers y_k with db_k != 0) or rows (labels x_k with dc_k != 0) into shared
// memory in ascending order, and every thread folds them into its own row or column.  The f update's reads are
// coalesced across threads; the b update's are strided by a row.  No workspace.
#include "spx_launch.cuh"

namespace {

using namespace spx;

constexpr int WARM_THREADS = 256;

struct WarmJob {
    double        *T;
    const int32_t *rowlab, *collab;
    const double  *db, *dc;              // either may be null; then its tiles are not launched
    int            n, m;                 // uniform batches
    const RaggedLp *lps;                 // ragged batches: LP order[q] for q < count, else uniform
    const int32_t  *order;
    int64_t        count;
    int            tb;                   // row tiles of the b update (0 when db is null)
};

// the ascending list of the chunk's active entries (act, idx, d) in s_idx / s_del; returns its length
__device__ __forceinline__ int block_compact(bool act, int idx, double d, int *s_idx, double *s_del, int *s_warp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned ball = __ballot_sync(0xffffffffu, act);
    if (lane == 0) s_warp[warp] = __popc(ball);
    __syncthreads();
    int base = 0, total = 0;
#pragma unroll
    for (int w = 0; w < WARM_THREADS / 32; ++w) {
        const int c = s_warp[w];
        base += (w < warp) ? c : 0;
        total += c;
    }
    if (act) {
        const int p = base + __popc(ball & ((1u << lane) - 1u));
        s_idx[p] = idx;
        s_del[p] = d;
    }
    __syncthreads();
    return total;
}

__global__ void __launch_bounds__(WARM_THREADS) warm_change_kernel(WarmJob J) {
    __shared__ int s_idx[WARM_THREADS];
    __shared__ double s_del[WARM_THREADS];
    __shared__ int s_warp[WARM_THREADS / 32];
    const bool brow = (int)blockIdx.x < J.tb;
    const int tile = brow ? (int)blockIdx.x : (int)blockIdx.x - J.tb;
    const int tid = (int)threadIdx.x;
    for (int64_t q = blockIdx.y; q < J.count; q += gridDim.y) {
        int n = J.n, m = J.m;
        int64_t t, xm, xn;
        if (J.lps) {
            const RaggedLp d = J.lps[J.order[q]];
            n = d.n; m = d.m; t = d.t; xm = d.xm; xn = d.xn;
        } else {
            t = q * ((int64_t)n * (m + 1) + m); xm = q * m; xn = q * n;
        }
        const int64_t w1 = m + 1;
        double *T = J.T + t;
        const int32_t *rl = J.rowlab + xm, *cl = J.collab + xn;
        if (brow) {
            if (tile * WARM_THREADS >= n) continue;         // uniform over the CTA
            const double *db = J.db + xn;
            const int i = tile * WARM_THREADS + tid;
            double v = 0.0;
            if (i < n) {
                v = T[i * w1 + m];
                const int L = cl[i];
                if (L >= m && L - m < n) {
                    const double d = db[L - m];
                    if (d != 0.0) v = __dadd_rn(v, d);
                }
            }
            for (int j0 = 0; j0 < m; j0 += WARM_THREADS) {
                const int j = j0 + tid;
                bool act = false;
                double d = 0.0;
                if (j < m) {
                    const int H = rl[j];
                    if (H >= m && H - m < n) { d = db[H - m]; act = (d != 0.0); }
                }
                const int cnt = block_compact(act, j, d, s_idx, s_del, s_warp);
                if (i < n) {
                    const double *row = T + i * w1;
                    for (int u = 0; u < cnt; ++u) v = __dsub_rn(v, __dmul_rn(s_del[u], row[s_idx[u]]));
                }
                __syncthreads();                            // the list is read before the next chunk's
            }
            if (i < n) T[i * w1 + m] = v;
        } else {
            if (tile * WARM_THREADS >= m) continue;
            const double *dc = J.dc + xm;
            const int j = tile * WARM_THREADS + tid;
            double *frow = T + (int64_t)n * w1;
            double v = 0.0;
            if (j < m) {
                v = frow[j];
                const int H = rl[j];
                if (H >= 0 && H < m) {
                    const double d = dc[H];
                    if (d != 0.0) v = __dadd_rn(v, d);
                }
            }
            for (int i0 = 0; i0 < n; i0 += WARM_THREADS) {
                const int i = i0 + tid;
                bool act = false;
                double d = 0.0;
                if (i < n) {
                    const int L = cl[i];
                    if (L >= 0 && L < m) { d = dc[L]; act = (d != 0.0); }
                }
                const int cnt = block_compact(act, i, d, s_idx, s_del, s_warp);
                if (j < m)
                    for (int u = 0; u < cnt; ++u) v = __dadd_rn(v, __dmul_rn(s_del[u], T[s_idx[u] * w1 + j]));
                __syncthreads();
            }
            if (j < m) frow[j] = v;
        }
    }
}

cudaError_t warm_launch(WarmJob J, int64_t max_n, int64_t max_m, cudaStream_t s) {
    if (J.count <= 0 || (!J.db && !J.dc)) return cudaSuccess;
    const int64_t tb = J.db ? (max_n + WARM_THREADS - 1) / WARM_THREADS : 0;
    const int64_t tf = J.dc ? (max_m + WARM_THREADS - 1) / WARM_THREADS : 0;
    if (tb + tf > INT32_MAX) return cudaErrorInvalidConfiguration;
    J.tb = (int)tb;
    const unsigned gy = (unsigned)(J.count < 65535 ? J.count : 65535);
    warm_change_kernel<<<dim3((unsigned)(tb + tf), gy), WARM_THREADS, 0, s>>>(J);
    spx_host::count_launch();
    return cudaGetLastError();
}

} // namespace

namespace spx_launch {

cudaError_t warm_change_uniform(double *T, int64_t B, int n, int m, const int32_t *rowlab, const int32_t *collab,
                                const double *db, const double *dc, cudaStream_t s) {
    WarmJob J{T, rowlab, collab, db, dc, n, m, nullptr, nullptr, B, 0};
    return warm_launch(J, n, m, s);
}

// one launch per launch of the plan, so LPs of like size share a grid (as the sensitivity report)
cudaError_t warm_change_ragged(const PlanView &v, double *T, const int32_t *rowlab, const int32_t *collab,
                               const double *db, const double *dc, cudaStream_t s) {
    for (int q = 0; q < v.P->nlaunch; ++q) {
        const RaggedLaunch &l = v.P->launch[q];
        WarmJob J{T, rowlab, collab, db, dc, 0, 0, v.d_lps, v.d_order + l.first, l.count, 0};
        const cudaError_t e = warm_launch(J, launch_max(v, l, [](const RaggedLp &d) { return d.n; }),
                                          launch_max(v, l, [](const RaggedLp &d) { return d.m; }), s);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

} // namespace spx_launch
