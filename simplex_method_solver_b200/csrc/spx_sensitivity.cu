// spx_sensitivity.cu — the sensitivity report of an optimal final table: shadow prices, slacks, reduced costs and the
// allowable ranges of every right-hand side and objective coefficient (spx_sensitivity_*, include/spx_b200.h).
//
// The final table is a dictionary (recalculate_matrix, simplex.py:143-177): x_B = b + T x_N, f = f0 + sum_j d_j x_N.
// Every output is either a copy of one cell chosen by the labels, or a minimum over separately rounded quotients of
// cells: for a column j labelled y_k, over its rows (rhs ranges); for a row i labelled x_k, over its columns (cost
// ranges).  A minimum does not depend on the order of reduction, so the tiles below meet through atomicMin on the bit
// patterns of non-negative doubles and the result equals a sequential statement bit for bit.
//
// Two launches per group of LPs, in order on the caller's stream:
//   sens_init_kernel  one thread per row and per column of each LP: the copies, +inf in every end that the tile kernel
//                     min-reduces, and NaN everywhere for an LP that is not optimal;
//   sens_tile_kernel  one CTA per tile of (row band x column range) of each optimal LP; a thread keeps the partial
//                     minima of its column across its rows, each row's quotients are min-reduced over a warp segment,
//                     and both meet the other tiles' in global memory through atomicMin.
#include <cstdint>

#include "spx_launch.cuh"

namespace {

constexpr int SENS_THREADS = 256;
constexpr int SENS_ROWS_PER_THREAD = 16;   // rows of a tile per thread: 16 * 256 / CW rows per tile
constexpr int SENS_UNROLL = 4;             // cells a thread loads before it divides
constexpr uint64_t SENS_INF_BITS = 0x7FF0000000000000ull;

enum SensLayout { SENS_UNIFORM = 0, SENS_RAGGED = 1, SENS_SPLIT = 2 };

// One group of LPs and every pointer the two kernels need; passed by value.
struct SensJob {
    int32_t layout;
    int32_t n, m;                  // SENS_UNIFORM, SENS_SPLIT
    int32_t cw;                    // tile columns: a power of two in 1..256
    int32_t split_optimal;         // SENS_SPLIT: the host's optimality test of the table
    const double *T;               // flat tables, or the split body A[(n+1)][ld]
    const double *b;               // SENS_SPLIT: b[n]
    int64_t ld;                    // SENS_SPLIT
    const spx::RaggedLp *lps;      // SENS_RAGGED: descriptors (device copy of the plan)
    const int32_t *order;          // SENS_RAGGED: LP indices of the plan, grouped by launch
    int64_t first, count;          // LPs order[first .. first+count) (SENS_RAGGED), else 0 .. count
    const int32_t *status;         // [B]; NULL for SENS_SPLIT
    const int32_t *rowlab, *collab;
    double *dual, *slack, *redcost, *rhs, *cost;
};

// One LP of a job: where its cells, labels and outputs are.
struct SensLp {
    const double *body;            // T[i][j] = body[i * pitch + j]
    int64_t pitch;
    const double *b;               // b_i = b[i * bstride]
    int64_t bstride;
    const double *f;               // d_j = f[j]
    const int32_t *rowlab, *collab;
    int64_t on, om;                // offsets of the per-constraint and the per-variable outputs
    int32_t n, m;
    bool optimal;
};

__device__ __forceinline__ SensLp sens_lp(const SensJob &J, int64_t s) {
    SensLp L;
    if (J.layout == SENS_SPLIT) {
        L.n = J.n; L.m = J.m;
        L.body = J.T; L.pitch = J.ld; L.b = J.b; L.bstride = 1; L.f = J.T + (int64_t)J.n * J.ld;
        L.rowlab = J.rowlab; L.collab = J.collab; L.on = 0; L.om = 0;
        L.optimal = J.split_optimal != 0;
        return L;
    }
    int64_t k, t, xm, xn;
    if (J.layout == SENS_RAGGED) {
        k = J.order[J.first + s];
        const spx::RaggedLp d = J.lps[k];
        L.n = d.n; L.m = d.m; t = d.t; xm = d.xm; xn = d.xn;
    } else {
        k = s;
        L.n = J.n; L.m = J.m;
        t = k * ((int64_t)J.n * (J.m + 1) + J.m); xm = k * J.m; xn = k * J.n;
    }
    L.body = J.T + t; L.pitch = L.m + 1; L.b = L.body + L.m; L.bstride = L.m + 1;
    L.f = L.body + (int64_t)L.n * (L.m + 1);
    L.rowlab = J.rowlab + xm; L.collab = J.collab + xn; L.on = xn; L.om = xm;
    L.optimal = J.status[k] == SPX_OPTIMAL;
    return L;
}

// every output zero is +0.0
__device__ __forceinline__ double pos0(double v) { return v == 0.0 ? 0.0 : v; }

__device__ __forceinline__ void put(double *p, int64_t i, double v) { if (p) p[i] = v; }
__device__ __forceinline__ void put2(double *p, int64_t i, double lo, double hi) {
    if (p) { p[2 * i] = lo; p[2 * i + 1] = hi; }
}

// grid (elements of the largest LP / 256, LPs); element e < n is body row e, else column e - n
__global__ void __launch_bounds__(SENS_THREADS) sens_init_kernel(SensJob J) {
    const double inf = __longlong_as_double((long long)SENS_INF_BITS);
    for (int64_t s = blockIdx.y; s < J.count; s += gridDim.y) {
        const SensLp L = sens_lp(J, s);
        const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (e >= (int64_t)L.n + L.m) continue;
        const int64_t nm = (int64_t)L.n + L.m;
        if (!L.optimal) {        // by position, whatever the labels hold
            const double nan = __longlong_as_double(0x7FF8000000000000ll);
            if (e < L.n) {
                put(J.dual, L.on + e, nan); put(J.slack, L.on + e, nan); put2(J.rhs, L.on + e, nan, nan);
            } else {
                put(J.redcost, L.om + e - L.n, nan); put2(J.cost, L.om + e - L.n, nan, nan);
            }
            continue;
        }
        if (e < L.n) {           // the row of basic variable collab[e] = b_e + ...
            const int32_t lab = L.collab[e];
            if (lab < 0 || lab >= nm) continue;
            const double bi = pos0(L.b[e * L.bstride]);
            if (lab >= L.m) {
                const int64_t k = L.on + (lab - L.m);
                put(J.dual, k, 0.0); put(J.slack, k, bi); put2(J.rhs, k, bi, inf);
            } else {
                const int64_t k = L.om + lab;
                put(J.redcost, k, 0.0); put2(J.cost, k, inf, inf);
            }
        } else {                 // the column of nonbasic variable rowlab[j]
            const int64_t j = e - L.n;
            const int32_t lab = L.rowlab[j];
            if (lab < 0 || lab >= nm) continue;
            const double d = L.f[j];
            if (lab >= L.m) {
                const int64_t k = L.on + (lab - L.m);
                put(J.dual, k, pos0(-d)); put(J.slack, k, 0.0); put2(J.rhs, k, inf, inf);
            } else {
                const int64_t k = L.om + lab;
                put(J.redcost, k, pos0(d)); put2(J.cost, k, pos0(d), inf);
            }
        }
    }
}

__device__ __forceinline__ void min_into(double *p, int64_t i, double v) {
    if (v < __longlong_as_double((long long)SENS_INF_BITS))     // +inf is already there; NaN never wins
        atomicMin(reinterpret_cast<unsigned long long *>(p) + i,
                  (unsigned long long)__double_as_longlong(pos0(v)));
}

// grid (tiles of the largest LP, LPs).  A tile is CW columns x (16 * 256 / CW) rows; thread t takes column t % CW and
// rows g, g + G, ... of the band, g = t / CW, G = 256 / CW.  All threads run the same number of row steps, so the
// segmented shuffles below always have every lane.
__global__ void __launch_bounds__(SENS_THREADS) sens_tile_kernel(SensJob J) {
    const double inf = __longlong_as_double((long long)SENS_INF_BITS);
    const int CW = J.cw, G = SENS_THREADS / CW, W = CW < 32 ? CW : 32;
    const int RB = SENS_ROWS_PER_THREAD * G;
    for (int64_t s = blockIdx.y; s < J.count; s += gridDim.y) {
        const SensLp L = sens_lp(J, s);
        if (!L.optimal) continue;
        const int64_t tiles_c = (L.m + CW - 1) / CW;
        const int64_t tiles = (L.n + (int64_t)RB - 1) / RB * tiles_c;
        if ((int64_t)blockIdx.x >= tiles) continue;
        const int64_t i0 = (int64_t)blockIdx.x / tiles_c * RB + threadIdx.x / CW;
        const int64_t j = (int64_t)blockIdx.x % tiles_c * CW + threadIdx.x % CW;
        const bool colok = j < L.m;
        const int32_t clab = colok ? L.rowlab[j] : -1;
        const bool ycol = J.rhs && clab >= L.m && clab < (int64_t)L.n + L.m;
        const double d = colok ? L.f[j] : 0.0;
        double dec = inf, inc = inf;                        // this column's partial rhs range
        const double *col = L.body + j;
        for (int r0 = 0; r0 < SENS_ROWS_PER_THREAD; r0 += SENS_UNROLL) {
            double t[SENS_UNROLL], bi[SENS_UNROLL];
            int32_t rl[SENS_UNROLL];
#pragma unroll
            for (int u = 0; u < SENS_UNROLL; ++u) {
                const int64_t i = i0 + (int64_t)(r0 + u) * G;
                const bool ok = i < L.n;
                t[u] = (ok && colok) ? __ldg(col + i * L.pitch) : 0.0;
                bi[u] = (ok && ycol) ? __ldg(L.b + i * L.bstride) : 0.0;
                rl[u] = (ok && J.cost) ? __ldg(L.collab + i) : -1;
            }
#pragma unroll
            for (int u = 0; u < SENS_UNROLL; ++u) {
                if (ycol) {
                    if (t[u] < 0.0) { const double q = bi[u] / (-t[u]); if (q < dec) dec = q; }
                    else if (t[u] > 0.0) { const double q = bi[u] / t[u]; if (q < inc) inc = q; }
                }
                // the row of x_k: its cost range is a minimum over the row's columns
                const bool xrow = rl[u] >= 0 && rl[u] < L.m;
                if (__any_sync(0xffffffffu, xrow)) {
                    double lo = inf, hi = inf;      // a NaN quotient never wins: it stays +inf
                    if (xrow) {
                        if (t[u] > 0.0) { const double q = d / t[u]; if (q < lo) lo = q; }
                        else if (t[u] < 0.0) { const double q = d / (-t[u]); if (q < hi) hi = q; }
                    }
                    for (int o = W >> 1; o > 0; o >>= 1) {   // over the CW lanes of the row (one warp at most)
                        const double lo2 = __shfl_xor_sync(0xffffffffu, lo, o);
                        const double hi2 = __shfl_xor_sync(0xffffffffu, hi, o);
                        if (lo2 < lo) lo = lo2;
                        if (hi2 < hi) hi = hi2;
                    }
                    if (xrow && (threadIdx.x & (W - 1)) == 0) {
                        const int64_t k = L.om + rl[u];
                        min_into(J.cost, 2 * k, lo);
                        min_into(J.cost, 2 * k + 1, hi);
                    }
                }
            }
        }
        if (ycol) {
            const int64_t k = L.on + (clab - L.m);
            min_into(J.rhs, 2 * k, dec);
            min_into(J.rhs, 2 * k + 1, inc);
        }
    }
}

int sens_cw(int64_t m) {
    int cw = 1;
    while (cw < m && cw < SENS_THREADS) cw <<= 1;
    return cw;
}

cudaError_t sens_launch(SensJob J, int64_t max_n, int64_t max_m, cudaStream_t s) {
    if (J.count == 0) return cudaSuccess;
    J.cw = sens_cw(max_m);
    const unsigned gy = (unsigned)(J.count < 65535 ? J.count : 65535);
    const int64_t ix = (max_n + max_m + SENS_THREADS - 1) / SENS_THREADS;
    sens_init_kernel<<<dim3((unsigned)ix, gy), SENS_THREADS, 0, s>>>(J);
    spx_host::count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess || (!J.rhs && !J.cost)) return e;
    const int64_t rb = (int64_t)SENS_ROWS_PER_THREAD * (SENS_THREADS / J.cw);
    const int64_t tiles = (max_n + rb - 1) / rb * ((max_m + J.cw - 1) / J.cw);
    if (tiles > INT32_MAX) return cudaErrorInvalidConfiguration;
    sens_tile_kernel<<<dim3((unsigned)tiles, gy), SENS_THREADS, 0, s>>>(J);
    spx_host::count_launch();
    return cudaGetLastError();
}

SensJob sens_job(int layout, const int32_t *status, const int32_t *rowlab, const int32_t *collab, double *dual,
                 double *slack, double *redcost, double *rhs, double *cost) {
    SensJob J{};
    J.layout = layout;
    J.status = status; J.rowlab = rowlab; J.collab = collab;
    J.dual = dual; J.slack = slack; J.redcost = redcost; J.rhs = rhs; J.cost = cost;
    return J;
}

} // namespace

namespace spx_launch {

cudaError_t sensitivity_uniform(const double *d_T, int64_t B, int n, int m, const int32_t *d_status,
                                const int32_t *d_rowlab, const int32_t *d_collab, double *dual, double *slack,
                                double *redcost, double *rhs, double *cost, cudaStream_t s) {
    SensJob J = sens_job(SENS_UNIFORM, d_status, d_rowlab, d_collab, dual, slack, redcost, rhs, cost);
    J.T = d_T; J.n = n; J.m = m; J.count = B;
    return sens_launch(J, n, m, s);
}

// one pair of launches per launch of the plan, so LPs of like size share a grid
cudaError_t sensitivity_ragged(const spx::PlanView &v, const double *d_T, const int32_t *d_status,
                               const int32_t *d_rowlab, const int32_t *d_collab, double *dual, double *slack,
                               double *redcost, double *rhs, double *cost, cudaStream_t s) {
    for (int q = 0; q < v.P->nlaunch; ++q) {
        const spx::RaggedLaunch &l = v.P->launch[q];
        SensJob J = sens_job(SENS_RAGGED, d_status, d_rowlab, d_collab, dual, slack, redcost, rhs, cost);
        J.T = d_T; J.lps = v.d_lps; J.order = v.d_order; J.first = l.first; J.count = l.count;
        const cudaError_t e = sens_launch(J, spx::launch_max(v, l, [](const spx::RaggedLp &d) { return d.n; }),
                                          spx::launch_max(v, l, [](const spx::RaggedLp &d) { return d.m; }), s);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t sensitivity_split(const double *d_A, const double *d_b, int n, int m, int64_t ld, int optimal,
                              const int32_t *d_rowlab, const int32_t *d_collab, double *dual, double *slack,
                              double *redcost, double *rhs, double *cost, cudaStream_t s) {
    SensJob J = sens_job(SENS_SPLIT, nullptr, d_rowlab, d_collab, dual, slack, redcost, rhs, cost);
    J.T = d_A; J.b = d_b; J.ld = ld; J.n = n; J.m = m; J.count = 1; J.split_optimal = optimal;
    return sens_launch(J, n, m, s);
}

} // namespace spx_launch
