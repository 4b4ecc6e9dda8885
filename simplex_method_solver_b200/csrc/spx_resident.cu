// spx_resident.cu — K5: the whole pivot loop as ONE persistent cooperative kernel for tableaus
// that live in the 126 MB L2 (cfg2: 1000 x 2000 = 2 x 16 MB): get_solution()'s loop,
// /root/reference/src/simplex.py:179-199, with pick_element() (:70-141) and
// recalculate_matrix() (:143-177) inside.
//
// A tableau that fits L2 is latency-bound, not HBM-bound: one pivot streams in ~4 us, so two
// kernel launches per pivot (pick + update, ~25 us) dominate.  Here every SM keeps one 512-thread CTA
// resident for the whole solve (measured: 11.8 us/pivot at cfg2; two 256-thread CTAs per SM: 13.9 —
// half as many redundant pricings hammer the same L2 lines and the barrier has half the arrivals)
// and a pivot costs ONE grid barrier:
//   - every CTA prices the pivot REDUNDANTLY (the decision depends on O(n + m) cells: its own
//     shared-memory replica of the b column, one row scan and one column gather from L2), so all
//     CTAs agree on (r, c, p) without exchanging anything;
//   - the CTAs then update their slices (a column tile of 512 x a band of rows, 128-bit accesses,
//     every row of the band in flight before the first division, L1 bypassed with
//     ld.global.cg / st.global.cg because other SMs wrote the lines one pivot earlier), every CTA
//     updates its replica of b, CTA 0 swaps the labels and appends to the trace;
//   - grid.sync(), swap the ping-pong buffers, next pivot.
// Arithmetic, selection rules and results are those of the streaming kernels (same helpers).
#include <cooperative_groups.h>

#include <cstdlib>

#include "spx_block.cuh"
#include "spx_launch.cuh"

namespace cg = cooperative_groups;

namespace {

using namespace spx;

constexpr int RES_THREADS = 512;
constexpr int RES_TC      = 2 * RES_THREADS;   // 1024 columns per tile
constexpr int RES_PASS    = 16;                // rows a thread keeps in flight per pass
constexpr int RES_MAX_N   = 4095;              // s_col + s_b must fit shared memory

struct ResidentArgs {
    double  *A[2];
    double  *b[2];
    int      n, m;
    int64_t  ld;
    int      rule;
    int64_t  max_steps;       // pivots to apply in this launch at most
    spx_state *st;
    double  *colbuf;          // receives the priced pivot column at exit (step API / look-ahead resume)
    int32_t *rowlab, *collab, *trace;
};

// developer aid (spx_resident_debug): cycles per phase summed over the pivots of the last launch, [15] = pivots
constexpr int RES_DBG = 16;
__device__ unsigned long long g_res_dbg[RES_DBG];
// STAMPS = false: an empty object — the shipped instantiations carry no trace of the instrumentation (measured: even
// switched off at run time it cost the default kernel 6 %, 11.2 -> 11.9 us per pivot on cfg2)
template <bool STAMPS> struct PhaseClock {
    __device__ __forceinline__ void start(unsigned long long *, bool) {}
    __device__ __forceinline__ void mark(int) {}
    __device__ __forceinline__ void finish(unsigned long long) {}
};
template <> struct PhaseClock<true> {
    unsigned long long *acc;
    long long last;
    bool on;
    __device__ __forceinline__ void start(unsigned long long *shared_acc, bool enable) {
        acc = shared_acc; on = enable;
        if (on) { for (int k = 0; k < RES_DBG; ++k) acc[k] = 0ull; last = clock64(); }
    }
    __device__ __forceinline__ void mark(int k) {
        if (on) { const long long t = clock64(); acc[k] += (unsigned long long)(t - last); last = t; }
    }
    __device__ __forceinline__ void finish(unsigned long long pivots) {
        if (on) { acc[RES_DBG - 1] = pivots; for (int k = 0; k < RES_DBG; ++k) g_res_dbg[k] = acc[k]; }
    }
};

__device__ __forceinline__ double2 ldcg2(const double *p) { return __ldcg(reinterpret_cast<const double2 *>(p)); }
__device__ __forceinline__ void stcg2(double *p, double2 v) { __stcg(reinterpret_cast<double2 *>(p), v); }

template <bool STAMPS>
__global__ void __launch_bounds__(RES_THREADS, 1)
resident_loop_kernel(ResidentArgs a) {
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(16) double res_smem[];
    __shared__ Scratch s;
    const int n = a.n, m = a.m;
    const int64_t ld = a.ld;
    double *s_col = res_smem;                       // [n + 1] pivot column of the current table
    double *s_b   = res_smem + ((n + 1 + 1) & ~1);  // [n]     this CTA's replica of the '-b' column
    const int tid = threadIdx.x, nt = blockDim.x;

    int64_t npiv = a.st->npiv;
    const int64_t cap = a.st->max_pivots;
    if (a.st->status != SPX_PIVOT) return;          // uniform over the grid: nobody reaches a barrier
    int cur = (int)(npiv & 1);
    for (int i = tid; i < n; i += nt) s_b[i] = __ldcg(a.b[cur] + i);
    __syncthreads();

    const int n_ct = (m + RES_TC - 1) / RES_TC;

    int status = SPX_PIVOT, r = -1, r1 = -1, cl = SPX_NONE;
    double p = 0.0;
    int64_t steps = 0;
    __shared__ unsigned long long s_acc[STAMPS ? RES_DBG : 1];
    PhaseClock<STAMPS> pc; pc.start(s_acc, blockIdx.x == 0 && tid == 0);
    for (;;) {
        pc.mark(0);                                        // (loop overhead, exit checks)
        const double *A = a.A[cur];
        double *An = a.A[cur ^ 1];
        // ---------------- K1: phase-1 row from the replica of b and, in the same sweep and the same
        // reduction, the first negative cell of the head of the f row (the two searches are independent;
        // the f head is what :94-98 finds in all but degenerate tables)
        const double *frow = A + (int64_t)n * ld;
        const int head = min(m, 4 * nt);
        int bneg = SPX_NONE, fneg = SPX_NONE;
        {
            double fv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { const int j = u * nt + tid; fv[u] = (j < head) ? __ldcg(frow + j) : 0.0; }
            for (int i = tid; i < n; i += nt) if (s_b[i] < 0.0) { bneg = i; break; }
#pragma unroll
            for (int u = 3; u >= 0; --u) { const int j = u * nt + tid; if (j < head && fv[u] < 0.0) fneg = j; }
        }
        pc.mark(1);                                        // b scan + f head loads
        block_min_int2(bneg, fneg, s);
        pc.mark(2);                                        // first reduction
        r1 = (bneg == SPX_NONE) ? -1 : bneg;
        if (r1 >= 0) {
            const double *row = A + (int64_t)r1 * ld;
            cl = block_first_index_fn(m, [&](int j) { return __ldcg(row + j); }, IsPos(), s);      // :82-85
        } else if (a.rule == SPX_RULE_REFERENCE) {
            cl = fneg;                                                                              // :94-98
            if (cl == SPX_NONE && m > head) {            // nothing in the head: scan the rest of the f row
                const int rest = block_first_index_fn(m - head, [&](int j) { return __ldcg(frow + head + j); }, IsNeg(), s);
                cl = (rest == SPX_NONE) ? SPX_NONE : head + rest;
            }
        } else {                                          // Dantzig: most negative, lowest index on ties
            const double *f = frow;
            unsigned long long best = ~0ull;
            for (int j = tid; j < m; j += nt) {
                const double v = __ldcg(f + j);
                if (v < 0.0) { const unsigned long long k = orderable(v); best = k < best ? k : best; }
            }
            best = block_min_u64(best, s);
            int loc = SPX_NONE;
            if (best != ~0ull)
                for (int j = tid; j < m; j += nt) {
                    const double v = __ldcg(f + j);
                    if (v < 0.0 && orderable(v) == best) { loc = j; break; }
                }
            cl = block_min_int(loc, s);
        }
        if (cl == SPX_NONE) {
            status = (r1 >= 0) ? SPX_INCORRECT : SPX_OPTIMAL;                                     // :88-89, :101-103
            break;
        }
        pc.mark(3);                                        // entering column decided
        // ---------------- K2: gather the column into shared memory, ratio test against the replica of b
        Ratio q = ratio_identity();
        for (int i = tid; i <= n; i += nt) {
            const double v = __ldcg(A + (int64_t)i * ld + cl);
            s_col[i] = v;
            if (r1 < 0 && i < n) ratio_accumulate(q, i, v, s_b[i]);
        }
        pc.mark(4);                                        // column gather + ratios
        if (r1 >= 0) {
            r = r1;                                                                               // :91
            __syncthreads();
        } else {
            q = block_ratio_reduce(q, s);                                                         // syncs: s_col is complete
            bool elig_nan = false;                        // a NaN ratio in the first eligible row is never replaced
            if (q.elig_row != SPX_NONE) {
                const double v = __ddiv_rn(s_b[q.elig_row], s_col[q.elig_row]);
                elig_nan = (v != v);
            }
            r = ratio_decide(q, elig_nan);                                                        // :138-141
            if (r < 0) { status = SPX_NOCONV; break; }
        }
        p = s_col[r];
        pc.mark(5);                                        // ratio reduction + decision
        if (npiv >= cap) { status = SPX_CAP; break; }
        if (steps >= a.max_steps) break;                   // priced, not applied: status stays SPX_PIVOT

        // ---------------- K3: this CTA's slice of the out-of-place update.  The CTAs are dealt out
        // as (column tile, row slice): a thread owns one column pair of the slice and loads ALL its
        // rows (up to RES_PASS per pass) before the first division — one L2 round trip per pivot.
        const PivotDiv d = pivot_div_prepare(p);
        const int per_ct = max(1, (int)gridDim.x / n_ct);          // CTAs that share one column tile
        for (int unit = blockIdx.x; unit < n_ct * per_ct; unit += gridDim.x) {
            const int ct = unit % n_ct, slice = unit / n_ct;
            const int j = ct * RES_TC + 2 * tid;
            if (j >= m) continue;
            const int rpc = (n + 1 + per_ct - 1) / per_ct;          // rows per CTA
            const int row_end = min(n + 1, (slice + 1) * rpc);
            const double2 rj = ldcg2(A + (int64_t)r * ld + j);
            const int jc = (cl >= j && cl < j + 2) ? cl - j : -1;
            for (int i0 = slice * rpc; i0 < row_end; i0 += RES_PASS) {
                double2 tv[RES_PASS];
#pragma unroll
                for (int u = 0; u < RES_PASS; ++u)
                    if (i0 + u < row_end) tv[u] = ldcg2(A + (int64_t)(i0 + u) * ld + j);
#pragma unroll
                for (int u = 0; u < RES_PASS; ++u)
                    if (i0 + u < row_end)
                        stcg2(An + (int64_t)(i0 + u) * ld + j,
                              generic_pair(tv[u], i0 + u, r, jc, rj, s_col[i0 + u], d));
            }
        }
        pc.mark(6);                                        // sweep (loads, arithmetic, stores issued)
        // ---------------- every CTA advances its replica of b (:155-156, :166-175 on the last column)
        const double br = s_b[r];
        __syncthreads();
        for (int i = tid; i < n; i += nt) {
            const double bi = s_b[i];
            s_b[i] = (i == r) ? pivot_div(-bi, d) : cell_update(bi, d, br, s_col[i]);
        }
        if (blockIdx.x == 0 && tid == 0) {                 // labels (:152) and the pivot trace
            const int32_t tmp = a.rowlab[cl]; a.rowlab[cl] = a.collab[r]; a.collab[r] = tmp;
            if (a.trace) { a.trace[2 * npiv] = r; a.trace[2 * npiv + 1] = cl; }
        }
        ++npiv; ++steps; cur ^= 1;
        pc.mark(7);                                        // b update, labels
        grid.sync();                                       // the new table is complete and visible in L2
        pc.mark(8);                                        // grid barrier
    }
    pc.finish((unsigned long long)steps);

    // ---------------- exit (uniform): CTA 0 publishes the state, the b column and the priced column
    if (blockIdx.x == 0) {
        __syncthreads();
        for (int i = tid; i < n; i += nt) a.b[cur][i] = s_b[i];
        if (status == SPX_PIVOT || status == SPX_CAP)
            for (int i = tid; i <= n; i += nt) a.colbuf[i] = s_col[i];
        if (tid == 0) {
            spx_state o;
            o.status = status; o.r = r; o.c = (cl == SPX_NONE) ? -1 : cl; o.p = p;
            o.npiv = npiv; o.max_pivots = cap; o.phase1 = (r1 >= 0) ? 1 : 0; o.slot = 0;
            o.hint_tag[0] = o.hint_tag[1] = -1;
            o.hint_bneg[0] = o.hint_bneg[1] = SPX_NONE;
            o.hint_fneg[0] = o.hint_fneg[1] = SPX_NONE;
            for (int k = 0; k < 6; ++k) o.reserved[k] = 0;
            *a.st = o;
        }
    }
}

int g_res_grid = -1;     // co-resident CTAs on this device (0: cooperative launch unsupported)

} // namespace

namespace spx_launch {

size_t resident_smem(int n) { return (size_t)(((n + 2) & ~1) + n + 2) * sizeof(double); }

// Can this tableau run in the resident loop?  (fits the shared-memory replicas and ~L2)
bool resident_fits(int n, int m, int64_t ld) {
    (void)m;
    if (n > RES_MAX_N) return false;
    if (2LL * (n + 1) * ld * 8 > (96LL << 20)) return false;
    if (g_res_grid < 0) {
        int dev = 0, coop = 0, per_sm = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        g_res_grid = 0;
        if (coop) {
            cudaFuncSetAttribute(resident_loop_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)resident_smem(RES_MAX_N));
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, resident_loop_kernel<false>, RES_THREADS,
                                                              resident_smem(RES_MAX_N)) == cudaSuccess && per_sm > 0)
                g_res_grid = per_sm * sm_count();
        }
    }
    static bool attr_dev[64] = {};                           // the dynamic shared-memory limit is a per-device attribute
    bool &attr = attr_dev[spx_host::device_slot()];
    if (g_res_grid > 0 && !attr) {
        cudaFuncSetAttribute(resident_loop_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)resident_smem(RES_MAX_N));
        cudaFuncSetAttribute(resident_loop_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)resident_smem(RES_MAX_N));
        attr = true;
    }
    return g_res_grid > 0;
}

// Apply at most `max_steps` pivots in one persistent launch; the outcome is in *st.
cudaError_t resident_loop(double *A0, double *A1, double *b0, double *b1, int n, int m, int64_t ld, int rule,
                          int64_t max_steps, spx_state *st, double *colbuf, int32_t *rowlab, int32_t *collab,
                          int32_t *trace, cudaStream_t stream) {
    if (!resident_fits(n, m, ld)) return cudaErrorNotSupported;
    ResidentArgs a;
    a.A[0] = A0; a.A[1] = A1; a.b[0] = b0; a.b[1] = b1;
    a.n = n; a.m = m; a.ld = ld; a.rule = rule; a.max_steps = max_steps;
    a.st = st; a.colbuf = colbuf; a.rowlab = rowlab; a.collab = collab; a.trace = trace;
    static const bool stamps = getenv("SPX_RESIDENT_STAMPS") != nullptr;      // developer aid: the instrumented instantiations
    // no more CTAs than (column tiles) x (rows): every CTA must own at least one row of one tile
    const int64_t n_ct = ((int64_t)m + RES_TC - 1) / RES_TC;
    const int64_t units = n_ct * ((int64_t)n + 1);
    int grid = g_res_grid;
    if (units < grid) grid = (int)units;
    if (grid < 1) grid = 1;
    void *args[] = {&a};
    const cudaError_t e = cudaLaunchCooperativeKernel(
        stamps ? (const void *)resident_loop_kernel<true> : (const void *)resident_loop_kernel<false>, dim3(grid),
        dim3(RES_THREADS), args, resident_smem(n), stream);
    spx_host::count_launch();
    return e;
}

// developer aid: the per-phase cycle sums of the last resident launch (SPX_RESIDENT_STAMPS=1), 16 values
cudaError_t resident_debug(unsigned long long *h_out) {
    return cudaMemcpyFromSymbol(h_out, g_res_dbg, sizeof(unsigned long long) * RES_DBG);
}

} // namespace spx_launch

extern "C" int spx_resident_debug(uint64_t *h_out16) {
    if (!h_out16) return -2;
    return spx_host::check(spx_launch::resident_debug(reinterpret_cast<unsigned long long *>(h_out16)), "resident debug");
}
