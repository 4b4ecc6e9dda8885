// spx_certificate.cu — certificates of the two failures, read off the final table (spx_certificate_*,
// include/spx_b200.h): the Farkas vector of an infeasible LP and the unbounded ray of an unbounded one.
//
// The final table is the dictionary x_B = b + T x_N, f = f0 + sum_j d_j x_N.  A row with b_r < 0 and no positive
// cell proves the LP infeasible; in a table with every b_i >= 0, a column with d_c < 0 and no negative cell is a ray
// along which f falls without bound.  The report is the lowest such row and the lowest such column, with the row and
// the column scattered by the labels.  Every step is a minimum of indices, a logical OR or a copy, so the kernels
// equal the sequential statement (tests/certificate_oracle.c) bit for bit on any grid.
//
// Three launches per group of LPs, in order on the caller's stream.  farkas [n] and ray [m] of each LP are the
// workspace: until the finishing pass they hold one flag word per row and per column, 0 while the row (column) is
// still a candidate, else 1.
//   cert_init_kernel    one team per LP (a warp, or a CTA for large LPs): row i is a candidate when b_i is finite
//                       and < 0; column j when every b_i is finite and >= 0 (a team-wide OR) and d_j is finite and
//                       < 0;
//   cert_tile_kernel    the tiles of sens_tile_kernel; a thread reads a cell only when its row or its column is still
//                       a candidate, and a row (column) with a cell that is positive (negative) or not finite is
//                       disqualified with an atomic OR.  On an optimal table nothing but the flags is read;
//   cert_finish_kernel  one team per LP: the lowest row (column) still a candidate by a team-wide atomicMin, then the
//                       row (column) is gathered and scattered by the labels.  A label that appears twice is resolved
//                       as the statement's sequential loop resolves it (the last writer wins) through an atomicMax of
//                       writer indices in the output itself.
#include <cfloat>
#include <climits>
#include <cstdint>

#include "spx_launch.cuh"

namespace {

constexpr int CERT_THREADS = 256;           // tile pass
constexpr int CERT_ROWS_PER_THREAD = 16;    // rows of a tile per thread: 16 * 256 / CW rows per tile
constexpr int CERT_UNROLL = 4;
constexpr int CERT_CTA_TEAM = 1024;         // init and finish: one CTA of 1024 threads per LP ...
constexpr int CERT_WARP_MAX = 1024;         // ... unless n + m <= 1024, then one warp per LP (8 per CTA)

enum CertLayout { CERT_UNIFORM = 0, CERT_RAGGED = 1, CERT_SPLIT = 2 };

typedef unsigned long long u64;

// One group of LPs and every pointer the three kernels need; passed by value.
struct CertJob {
    int32_t layout;
    int32_t n, m;                  // CERT_UNIFORM, CERT_SPLIT
    int32_t cw;                    // tile columns: a power of two in 1..256
    const double *T;               // flat tables, or the split body A[(n+1)][ld]
    const double *b;               // CERT_SPLIT: b[n]
    int64_t ld;                    // CERT_SPLIT
    const spx::RaggedLp *lps;      // CERT_RAGGED: descriptors (device copy of the plan)
    const int32_t *order;          // CERT_RAGGED: LP indices of the plan, grouped by launch
    int64_t first, count;          // LPs order[first .. first+count) (CERT_RAGGED), else 0 .. count
    const int32_t *rowlab, *collab;
    int32_t *row;
    double *farkas, *bound;        // farkas == NULL: no Farkas half (row and bound are NULL too)
    int32_t *col;
    double *ray, *slope;           // ray == NULL: no ray half (col and slope are NULL too)
};

// One LP of a job: where its cells, labels and outputs are.
struct CertLp {
    const double *body;            // T[i][j] = body[i * pitch + j]
    int64_t pitch;
    const double *b;               // b_i = b[i * bstride]
    int64_t bstride;
    const double *f;               // d_j = f[j]
    const int32_t *rowlab, *collab;
    int64_t on, om, k;             // offsets of the per-constraint and per-variable outputs, index of the LP
    int32_t n, m;
};

__device__ __forceinline__ CertLp cert_lp(const CertJob &J, int64_t s) {
    CertLp L;
    if (J.layout == CERT_SPLIT) {
        L.n = J.n; L.m = J.m;
        L.body = J.T; L.pitch = J.ld; L.b = J.b; L.bstride = 1; L.f = J.T + (int64_t)J.n * J.ld;
        L.rowlab = J.rowlab; L.collab = J.collab; L.on = 0; L.om = 0; L.k = 0;
        return L;
    }
    int64_t t, xm, xn;
    if (J.layout == CERT_RAGGED) {
        L.k = J.order[J.first + s];
        const spx::RaggedLp d = J.lps[L.k];
        L.n = d.n; L.m = d.m; t = d.t; xm = d.xm; xn = d.xn;
    } else {
        L.k = s;
        L.n = J.n; L.m = J.m;
        t = s * ((int64_t)J.n * (J.m + 1) + J.m); xm = s * J.m; xn = s * J.n;
    }
    L.body = J.T + t; L.pitch = L.m + 1; L.b = L.body + L.m; L.bstride = L.m + 1;
    L.f = L.body + (int64_t)L.n * (L.m + 1);
    L.rowlab = J.rowlab + xm; L.collab = J.collab + xn; L.on = xn; L.om = xm;
    return L;
}

__device__ __forceinline__ bool neg_finite(double v) { return v < 0.0 && v >= -DBL_MAX; }
__device__ __forceinline__ bool nonpos_finite(double v) { return v <= 0.0 && v >= -DBL_MAX; }
__device__ __forceinline__ bool nonneg_finite(double v) { return v >= 0.0 && v <= DBL_MAX; }

// the flag words of an LP (the workspace in farkas and ray); NULL when that half is not computed
__device__ __forceinline__ u64 *row_flags(const CertJob &J, const CertLp &L) {
    return J.farkas ? reinterpret_cast<u64 *>(J.farkas + L.on) : nullptr;
}
__device__ __forceinline__ u64 *col_flags(const CertJob &J, const CertLp &L) {
    return J.ray ? reinterpret_cast<u64 *>(J.ray + L.om) : nullptr;
}

// A team is a warp (TEAM = 32, blocks of 256) or the whole CTA (TEAM = 1024).
template <int TEAM> __device__ __forceinline__ void team_sync() {
    if (TEAM == 32) __syncwarp(); else __syncthreads();
}
template <int TEAM> __device__ __forceinline__ bool team_any(bool p) {
    return TEAM == 32 ? __any_sync(0xffffffffu, p) : __syncthreads_or(p) != 0;
}
// the least v over the team (INT_MAX: none)
template <int TEAM> __device__ __forceinline__ int team_min(int v, int *s_min) {
    if (TEAM == 32) return __reduce_min_sync(0xffffffffu, v);
    if (threadIdx.x == 0) *s_min = INT_MAX;
    __syncthreads();
    if (v != INT_MAX) atomicMin(s_min, v);
    __syncthreads();
    const int r = *s_min;
    __syncthreads();
    return r;
}

// grid: teams over LPs
template <int TEAM> __global__ void __launch_bounds__(TEAM == 32 ? 256 : TEAM) cert_init_kernel(CertJob J) {
    const int per = blockDim.x / TEAM, t = threadIdx.x % TEAM;
    for (int64_t s = (int64_t)blockIdx.x * per + threadIdx.x / TEAM; s < J.count; s += (int64_t)gridDim.x * per) {
        const CertLp L = cert_lp(J, s);
        u64 *rf = row_flags(J, L), *cf = col_flags(J, L);
        bool bad = false;                               // some b_i is not finite and >= 0
        for (int i = t; i < L.n; i += TEAM) {
            const double bi = L.b[(int64_t)i * L.bstride];
            bad |= !nonneg_finite(bi);
            if (rf) rf[i] = neg_finite(bi) ? 0ull : 1ull;
        }
        if (cf) {
            const bool feasible = !team_any<TEAM>(bad);
            for (int j = t; j < L.m; j += TEAM) cf[j] = (feasible && neg_finite(L.f[j])) ? 0ull : 1ull;
        }
    }
}

__device__ __forceinline__ bool candidate(const u64 *flags, int64_t i) {
    return *reinterpret_cast<const volatile u64 *>(flags + i) == 0ull;    // other CTAs may be disqualifying it
}

// grid (tiles of the largest LP, LPs).  A tile is CW columns x (16 * 256 / CW) rows; thread t takes column t % CW and
// rows g, g + G, ... of the band, g = t / CW, G = 256 / CW.  All threads run the same number of row steps, so the
// segmented ballots below always have every lane.
__global__ void __launch_bounds__(CERT_THREADS) cert_tile_kernel(CertJob J) {
    const int CW = J.cw, G = CERT_THREADS / CW, W = CW < 32 ? CW : 32;
    const int RB = CERT_ROWS_PER_THREAD * G;
    const int lane = threadIdx.x & 31, seg = lane & ~(W - 1);
    const unsigned segmask = W == 32 ? 0xffffffffu : ((1u << W) - 1u);
    for (int64_t s = blockIdx.y; s < J.count; s += gridDim.y) {
        const CertLp L = cert_lp(J, s);
        const int64_t tiles_c = (L.m + CW - 1) / CW;
        const int64_t tiles = (L.n + (int64_t)RB - 1) / RB * tiles_c;
        if ((int64_t)blockIdx.x >= tiles) continue;
        u64 *rf = row_flags(J, L), *cf = col_flags(J, L);
        const int64_t i0 = (int64_t)blockIdx.x / tiles_c * RB + threadIdx.x / CW;
        const int64_t j = (int64_t)blockIdx.x % tiles_c * CW + threadIdx.x % CW;
        const bool colok = j < L.m;
        const bool ccand = colok && cf && candidate(cf, j);
        bool cbad = false;                              // this column has a negative or non-finite cell
        const double *col = L.body + j;
        for (int r0 = 0; r0 < CERT_ROWS_PER_THREAD; r0 += CERT_UNROLL) {
            double t[CERT_UNROLL];
            bool rc[CERT_UNROLL], ok[CERT_UNROLL];
#pragma unroll
            for (int u = 0; u < CERT_UNROLL; ++u) {
                const int64_t i = i0 + (int64_t)(r0 + u) * G;
                ok[u] = i < L.n;
                rc[u] = ok[u] && rf && candidate(rf, i);
                t[u] = (ok[u] && colok && (rc[u] || ccand)) ? col[i * L.pitch] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < CERT_UNROLL; ++u) {
                if (ccand && ok[u]) cbad |= !nonneg_finite(t[u]);
                const unsigned bal = __ballot_sync(0xffffffffu, rc[u] && colok && !nonpos_finite(t[u]));
                if (rc[u] && lane == seg && ((bal >> seg) & segmask))         // one lane per row segment
                    atomicOr(rf + i0 + (int64_t)(r0 + u) * G, 1ull);
            }
        }
        if (ccand && cbad) atomicOr(cf + j, 1ull);
    }
}

// Finishing pass of one half: the lowest candidate still standing (or none), then out = +0.0, the basis label's
// 1.0 and the line's cells scattered by the labels.  Writers are ordered as in the statement (the basis label
// first, then the line's cells in ascending order), and each output word keeps the latest writer by an atomicMax
// of (its index + 2); a word nobody wrote stays 0, i.e. +0.0.
//   Farkas half: line = row r, lo..hi = y labels (out index = label - m), cell q = 0.0 - T[r][q] for column q
//   ray half:    line = column c, lo..hi = x labels (out index = label), cell q = T[q][c] + 0.0 for row q
template <int TEAM, bool FARKAS>
__device__ __forceinline__ void cert_finish(const CertJob &J, const CertLp &L, int *s_min) {
    double *out = FARKAS ? J.farkas + L.on : J.ray + L.om;
    const int len = FARKAS ? L.n : L.m;                 // entries of the certificate = flag words
    const int lines = FARKAS ? L.m : L.n;               // cells of the row (column) scattered by the labels
    const int lo = FARKAS ? L.m : 0;
    const int t = threadIdx.x % TEAM;
    u64 *w = reinterpret_cast<u64 *>(out);
    int first = INT_MAX;
    for (int q = t; q < len; q += TEAM)
        if (w[q] == 0ull) { first = q; break; }
    const int r = team_min<TEAM>(first, s_min);
    team_sync<TEAM>();
    if (r == INT_MAX) {
        const double nan = __longlong_as_double(0x7FF8000000000000ll);
        for (int q = t; q < len; q += TEAM) out[q] = nan;
        if (t == 0) {
            if (FARKAS) { if (J.row) J.row[L.k] = -1; if (J.bound) J.bound[L.k] = nan; }
            else        { if (J.col) J.col[L.k] = -1; if (J.slope) J.slope[L.k] = nan; }
        }
        return;
    }
    for (int q = t; q < len; q += TEAM) w[q] = 0ull;
    team_sync<TEAM>();
    if (t == 0) {
        const int32_t lab = FARKAS ? L.collab[r] : L.rowlab[r];
        if (lab >= lo && lab - lo < len) atomicMax(w + (lab - lo), 1ull);
    }
    for (int q = t; q < lines; q += TEAM) {
        const int32_t lab = FARKAS ? L.rowlab[q] : L.collab[q];
        if (lab >= lo && lab - lo < len) atomicMax(w + (lab - lo), (u64)q + 2ull);
    }
    team_sync<TEAM>();
    for (int q = t; q < len; q += TEAM) {
        const u64 v = w[q];
        double x = 0.0;
        if (v == 1ull) {
            x = 1.0;
        } else if (v >= 2ull) {
            const int64_t p = (int64_t)(v - 2ull);
            x = FARKAS ? __dsub_rn(0.0, L.body[(int64_t)r * L.pitch + p]) : __dadd_rn(L.body[p * L.pitch + r], 0.0);
        }
        out[q] = x;
    }
    if (t == 0) {
        if (FARKAS) { if (J.row) J.row[L.k] = r; if (J.bound) J.bound[L.k] = L.b[(int64_t)r * L.bstride]; }
        else        { if (J.col) J.col[L.k] = r; if (J.slope) J.slope[L.k] = L.f[r]; }
    }
}

template <int TEAM> __global__ void __launch_bounds__(TEAM == 32 ? 256 : TEAM) cert_finish_kernel(CertJob J) {
    __shared__ int s_min;
    const int per = blockDim.x / TEAM;
    for (int64_t s = (int64_t)blockIdx.x * per + threadIdx.x / TEAM; s < J.count; s += (int64_t)gridDim.x * per) {
        const CertLp L = cert_lp(J, s);
        if (J.farkas) cert_finish<TEAM, true>(J, L, &s_min);
        team_sync<TEAM>();
        if (J.ray) cert_finish<TEAM, false>(J, L, &s_min);
        team_sync<TEAM>();
    }
}

int cert_cw(int64_t m) {
    int cw = 1;
    while (cw < m && cw < CERT_THREADS) cw <<= 1;
    return cw;
}

cudaError_t cert_launch(CertJob J, int64_t max_n, int64_t max_m, cudaStream_t s) {
    if (J.count == 0 || (!J.farkas && !J.ray)) return cudaSuccess;
    J.cw = cert_cw(max_m);
    const int64_t rb = (int64_t)CERT_ROWS_PER_THREAD * (CERT_THREADS / J.cw);
    const int64_t tiles = (max_n + rb - 1) / rb * ((max_m + J.cw - 1) / J.cw);
    if (tiles > INT32_MAX) return cudaErrorInvalidConfiguration;
    const bool warp = max_n + max_m <= CERT_WARP_MAX;
    const int64_t per = warp ? 256 / 32 : 1;
    const unsigned teams = (unsigned)((J.count + per - 1) / per < (1 << 20) ? (J.count + per - 1) / per : (1 << 20));
    if (warp) cert_init_kernel<32><<<teams, 256, 0, s>>>(J);
    else      cert_init_kernel<CERT_CTA_TEAM><<<teams, CERT_CTA_TEAM, 0, s>>>(J);
    spx_host::count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const unsigned gy = (unsigned)(J.count < 65535 ? J.count : 65535);
    cert_tile_kernel<<<dim3((unsigned)tiles, gy), CERT_THREADS, 0, s>>>(J);
    spx_host::count_launch();
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (warp) cert_finish_kernel<32><<<teams, 256, 0, s>>>(J);
    else      cert_finish_kernel<CERT_CTA_TEAM><<<teams, CERT_CTA_TEAM, 0, s>>>(J);
    spx_host::count_launch();
    return cudaGetLastError();
}

CertJob cert_job(int layout, const int32_t *rowlab, const int32_t *collab, int32_t *row, double *farkas,
                 double *bound, int32_t *col, double *ray, double *slope) {
    CertJob J{};
    J.layout = layout;
    J.rowlab = rowlab; J.collab = collab;
    J.row = row; J.farkas = farkas; J.bound = bound; J.col = col; J.ray = ray; J.slope = slope;
    return J;
}

} // namespace

namespace spx_launch {

cudaError_t certificate_uniform(const double *d_T, int64_t B, int n, int m, const int32_t *d_rowlab,
                                const int32_t *d_collab, int32_t *row, double *farkas, double *bound, int32_t *col,
                                double *ray, double *slope, cudaStream_t s) {
    CertJob J = cert_job(CERT_UNIFORM, d_rowlab, d_collab, row, farkas, bound, col, ray, slope);
    J.T = d_T; J.n = n; J.m = m; J.count = B;
    return cert_launch(J, n, m, s);
}

// one group of launches per launch of the plan, so LPs of like size share a grid
cudaError_t certificate_ragged(const spx::PlanView &v, const double *d_T, const int32_t *d_rowlab,
                               const int32_t *d_collab, int32_t *row, double *farkas, double *bound, int32_t *col,
                               double *ray, double *slope, cudaStream_t s) {
    for (int q = 0; q < v.P->nlaunch; ++q) {
        const spx::RaggedLaunch &l = v.P->launch[q];
        CertJob J = cert_job(CERT_RAGGED, d_rowlab, d_collab, row, farkas, bound, col, ray, slope);
        J.T = d_T; J.lps = v.d_lps; J.order = v.d_order; J.first = l.first; J.count = l.count;
        const cudaError_t e = cert_launch(J, spx::launch_max(v, l, [](const spx::RaggedLp &d) { return d.n; }),
                                          spx::launch_max(v, l, [](const spx::RaggedLp &d) { return d.m; }), s);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t certificate_split(const double *d_A, const double *d_b, int n, int m, int64_t ld,
                              const int32_t *d_rowlab, const int32_t *d_collab, int32_t *row, double *farkas,
                              double *bound, int32_t *col, double *ray, double *slope, cudaStream_t s) {
    CertJob J = cert_job(CERT_SPLIT, d_rowlab, d_collab, row, farkas, bound, col, ray, slope);
    J.T = d_A; J.b = d_b; J.ld = ld; J.n = n; J.m = m; J.count = 1;
    return cert_launch(J, n, m, s);
}

} // namespace spx_launch
