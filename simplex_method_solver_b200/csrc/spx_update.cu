// spx_update.cu — K3: the Gauss-Jordan / dictionary rank-1 update,
// recalculate_matrix(), /root/reference/src/simplex.py:149-177.
//
// Memory-bound fp64 stream: every body cell is read once (8 B) and written once
// (8 B) — the 16 B/cell/pivot of BASELINE.json — out of place between two
// ping-pong buffers, so there is no hazard and the pivot row/column are
// immutable for the whole pivot.  Per cell: 2 DMUL + 1 DADD for t*p - rj*ci and
// 1 DMUL + 2 DFMA for the division by the pivot (reciprocal hoisted, see
// pivot_div in spx_common.cuh) = 6 fp64 issues against 16 B of traffic.
//
// update_tiled_kernel: one CTA per tile of TR (default 8) rows x 512 columns; a thread
// owns two adjacent columns (one 128-bit access per row) and walks down the rows: fully
// coalesced 512-byte line groups, the thread's two pivot-row values in registers, the
// column multiplier a shared-memory broadcast.  The pivot-row slice and the pivot-column
// slice are staged with two cp.async.bulk (TMA, SASS UBLKCP) copies on one mbarrier.
// 8 rows in flight per thread, 4 CTAs per SM (64 registers): 6.8 TB/s at cfg4.
//
// Fused into the same pass: the b ('-b') column update, the label swap
// (:152), the pivot trace, and the pricing of the NEXT pivot (first negative
// new f / new b index, min-reduced into the state) so the next pick starts
// without scanning.
#include "spx_launch.cuh"

namespace {

using namespace spx;

constexpr int UPD_THREADS = 256;
constexpr int UPD_TC      = 2 * UPD_THREADS;   // columns per tile
constexpr int UPD_TR_MAX  = 64;                // rows per tile (upper bound; multiple of 8)
constexpr int UPD_UNROLL  = 8;

// the '-b' column (replicated when column-sharded) for rows [row_begin, row_end) + hint
__device__ __forceinline__ void update_b_rows(const double *__restrict__ bin, double *__restrict__ bout,
                                              const double *__restrict__ colbuf, int n, int r,
                                              const PivotDiv &d, int i, bool valid, int *hint) {
    int bneg = SPX_NONE;
    if (valid && i < n) {
        const double bi = bin[i];
        const double nb = (i == r) ? pivot_div(-bi, d) : cell_update(bi, d, bin[r], colbuf[i]);
        bout[i] = nb;
        if (nb < 0.0) bneg = i;
    }
    const int w = __reduce_min_sync(0xffffffffu, bneg);
    if ((threadIdx.x & 31) == 0 && w != SPX_NONE) atomicMin(hint, w);
}

// commit: labels (:152), trace, pivot counter — one thread of one CTA
// ahead != 0: the look-ahead kernels own the state and the b column (the next state is written
// by ahead_select_kernel while this kernel still reads the current one), so nothing is stored to *st
__device__ __forceinline__ void commit_pivot(spx_state *st, int r, int64_t cg, int slot,
                                             int32_t *rowlab, int32_t *collab, int32_t *trace, int ahead) {
    const int64_t k = st->npiv;
    const int32_t tmp = rowlab[cg]; rowlab[cg] = collab[r]; collab[r] = tmp;
    if (trace) { trace[2 * k] = r; trace[2 * k + 1] = (int32_t)cg; }
    if (!ahead) {
        st->hint_tag[slot] = k + 1;
        st->npiv = k + 1;
    }
}

template <int MINB>
__global__ void __launch_bounds__(UPD_THREADS, MINB)
update_tiled_kernel(const double *__restrict__ Ain, double *__restrict__ Aout,
                    const double *__restrict__ bin, double *__restrict__ bout,
                    int n, int m_loc, int64_t ld, int64_t col0, int tr, int ahead,
                    spx_state *st, const double *__restrict__ colbuf,
                    int32_t *__restrict__ rowlab, int32_t *__restrict__ collab,
                    int32_t *__restrict__ trace) {
    if (st->status != SPX_PIVOT) return;

    __shared__ alignas(128) double s_row[UPD_TC];
    __shared__ alignas(128) double s_col[UPD_TR_MAX];
    __shared__ alignas(8) uint64_t s_bar;

    const int     r    = st->r;
    const int64_t cg   = st->c;
    const int     slot = st->slot;
    const PivotDiv d   = pivot_div_prepare(st->p);

    const int tid  = threadIdx.x;
    const int j0   = blockIdx.x * UPD_TC;
    const int i0   = blockIdx.y * tr;
    const int rows = min(tr, n + 1 - i0);

    // ---- stage the pivot-row slice and the pivot-column slice (TMA bulk copies)
    const uint32_t row_bytes = (uint32_t)(min((int64_t)UPD_TC, ld - j0) * 8);   // ld % 16 == 0
    const uint32_t col_bytes = (uint32_t)(tr * 8);        // colbuf is padded to a whole tile
    if (tid == 0) {
        mbar_init(&s_bar, 1);
        mbar_fence_init();
        mbar_expect_tx(&s_bar, row_bytes + col_bytes);
        bulk_g2s(s_row, Ain + (int64_t)r * ld + j0, row_bytes, &s_bar);
        bulk_g2s(s_col, colbuf + i0, col_bytes, &s_bar);
    }
    __syncthreads();               // barrier init visible to the waiters
    mbar_wait(&s_bar, 0);

    const int  j      = j0 + 2 * tid;                    // local column of .x
    const bool active = j < m_loc;
    const int64_t cl   = cg - col0;                      // local index of the pivot column
    const bool has_c   = (cl >= j0) && (cl < j0 + UPD_TC);
    const int  jc      = has_c ? (int)(cl - j) : -1;
    const bool has_r   = (r >= i0) && (r < i0 + rows);
    const bool has_f   = (i0 + rows == n + 1);
    // CTA-uniform: interior tiles (no pivot row / pivot column / f row, full height)
    const bool plain   = !has_c && !has_r && !has_f && (rows % UPD_UNROLL == 0);

    int fneg = SPX_NONE;                                 // first negative new f index in this thread
    if (active) {
        const double2 rj = *reinterpret_cast<const double2 *>(&s_row[2 * tid]);
        const double *src = Ain + (int64_t)i0 * ld + j;
        double *dst = Aout + (int64_t)i0 * ld + j;
        if (plain) {
            for (int ii = 0; ii < rows; ii += UPD_UNROLL) {
                double2 t[UPD_UNROLL];
#pragma unroll
                for (int u = 0; u < UPD_UNROLL; ++u) t[u] = ld_stream(src + (int64_t)(ii + u) * ld);
#pragma unroll
                for (int u = 0; u < UPD_UNROLL; ++u) {
                    const double ci = s_col[ii + u];
                    double2 o;
                    o.x = cell_update(t[u].x, d, rj.x, ci);
                    o.y = cell_update(t[u].y, d, rj.y, ci);
                    st_stream(dst + (int64_t)(ii + u) * ld, o);
                }
            }
        } else {
            for (int ii = 0; ii < rows; ii += UPD_UNROLL) {
                double2 t[UPD_UNROLL];
#pragma unroll
                for (int u = 0; u < UPD_UNROLL; ++u)
                    if (ii + u < rows) t[u] = ld_stream(src + (int64_t)(ii + u) * ld);
#pragma unroll
                for (int u = 0; u < UPD_UNROLL; ++u) {
                    if (ii + u < rows) {
                        const int i = i0 + ii + u;
                        const double2 o = generic_pair(t[u], i, r, jc, rj, s_col[ii + u], d);
                        st_stream(dst + (int64_t)(ii + u) * ld, o);
                        if (i == n) {                                    // new f row: price the next pivot
                            if (o.x < 0.0) fneg = j;
                            else if (o.y < 0.0 && j + 1 < m_loc) fneg = j + 1;
                        }
                    }
                }
            }
        }
    }
    if (has_f && !ahead) {                               // this tile holds the f row (CTA-uniform)
        const int w = __reduce_min_sync(0xffffffffu, fneg);
        if ((tid & 31) == 0 && w != SPX_NONE) atomicMin(&st->hint_fneg[slot], w);
    }

    // ---- the '-b' column: column tile 0 does it
    if (blockIdx.x == 0) {
        if (tid < 64 && !ahead)                          // warps 0,1 cover tr <= 64 rows
            update_b_rows(bin, bout, colbuf, n, r, d, i0 + tid, tid < rows, &st->hint_bneg[slot]);
        if (blockIdx.y == 0 && tid == 0) commit_pivot(st, r, cg, slot, rowlab, collab, trace, ahead);
    }
}

// a / p for arrays: the self-test of pivot_div against the compiler's div.rn.f64
__global__ void division_selftest_kernel(const double *__restrict__ a, const double *__restrict__ p,
                                         int64_t count, int64_t np, unsigned long long *mismatches,
                                         double *first_bad) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < count;
         k += (int64_t)gridDim.x * blockDim.x) {
        const double pv = p[k % np];
        const PivotDiv d = pivot_div_prepare(pv);
        const double q = pivot_div(a[k], d);
        const double e = __ddiv_rn(a[k], pv);
        // pivot_div_unchecked: guards accumulated, exact redo when one tripped
        bool ok = true;
        double q2 = pivot_div_unchecked(a[k], d, ok);
        if (!ok) q2 = pivot_div(a[k], d);
        const bool same = ((__double_as_longlong(q) == __double_as_longlong(e)) || (q != q && e != e)) &&
                          ((__double_as_longlong(q2) == __double_as_longlong(e)) || (q2 != q2 && e != e));
        if (!same) {
            if (atomicAdd(mismatches, 1ull) == 0ull) { first_bad[0] = a[k]; first_bad[1] = pv; }
        }
    }
}

// find_optimum()/f(), simplex.py:48-68, for all m variables
__global__ void extract_kernel(const double *__restrict__ b, int n, int m,
                               const int32_t *__restrict__ collab,
                               const double *__restrict__ function,
                               double *__restrict__ x, double *__restrict__ obj) {
    // x is pre-zeroed by the launcher; labels are unique so the scatter is race-free
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int lab = collab[i];
        if (lab >= 0 && lab < m) x[lab] = b[i];
    }
}

__global__ void objective_kernel(int m, const double *__restrict__ function,
                                 const double *__restrict__ x, double *__restrict__ obj) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        obj[0] = (m >= 2) ? __dadd_rn(__dmul_rn(function[0], x[0]), __dmul_rn(function[1], x[1])) : 0.0;
        double s = 0.0;
        for (int j = 0; j < m; ++j) s = __dadd_rn(s, __dmul_rn(function[j], x[j]));
        obj[1] = s;
    }
}

__global__ void init_state_kernel(spx_state *st, int32_t *rowlab, int32_t *collab, int n, int m,
                                  int64_t max_pivots) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int stride = gridDim.x * blockDim.x;
    for (int j = t; j < m; j += stride) rowlab[j] = j;          // 'x1'..'xm'  :30
    for (int i = t; i < n; i += stride) collab[i] = m + i;      // 'y1'..'yn'  :31
    if (t == 0) {
        st->status = SPX_PIVOT; st->r = -1; st->c = -1; st->p = 0.0;
        st->npiv = 0; st->max_pivots = max_pivots; st->phase1 = 0; st->slot = 1;
        st->hint_tag[0] = -1; st->hint_tag[1] = -1;
        st->hint_bneg[0] = st->hint_bneg[1] = SPX_NONE;
        st->hint_fneg[0] = st->hint_fneg[1] = SPX_NONE;
        for (int q = 0; q < 6; ++q) st->reserved[q] = 0;
    }
}

int g_sm_count = 0;

} // namespace

namespace spx_launch {

int sm_count() {
    if (g_sm_count == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev);
        if (g_sm_count <= 0) g_sm_count = 148;
    }
    return g_sm_count;
}

int64_t colbuf_doubles(int n) {
    // whole row tiles for any tile height <= UPD_TR_MAX (the TMA copy reads a full tile)
    return ((int64_t)n + 1 + UPD_TR_MAX - 1) / UPD_TR_MAX * UPD_TR_MAX + UPD_TR_MAX;
}

int64_t g_opt[17] = {0, 0, 4, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};

// Rows per tile.  Measured on B200 (tools/upd_lab.py, profiles/r1c_update_variants.md): the smallest
// tile — 8 rows = exactly one 8-deep load batch per thread, 4 CTAs (64 registers) per SM — is the
// fastest at every size: 16384 x 32768 streams at 6.79 TB/s (64 rows: 6.60), and the 4096-column
// shard of the 8-GPU split at 5.9 TB/s (64 rows: 4.8, wave quantisation: 2056 CTAs on 444 slots).
static int pick_tr(int n, int m_loc) {
    (void)n; (void)m_loc;
    if (g_opt[SPX_OPT_TILED_ROWS] > 0) return (int)g_opt[SPX_OPT_TILED_ROWS];
    return 8;
}

// process-wide tuning knobs (spx_set_option); every setting computes the same bits

// SPX_OPT_FUSE_DEPTH reads the depth the one-GPU fused loop uses, the default included
int64_t get_option(int key) {
    if (key == SPX_OPT_FUSE_DEPTH && g_opt[key] == 0) return fuse_max();
    return (key >= 0 && key < 17) ? g_opt[key] : -1;
}
int set_option(int key, int64_t value) {
    switch (key) {
    case SPX_OPT_TILED_MIN_BLOCKS: if (value < 1 || value > 4) return -1; break;
    case SPX_OPT_TILED_ROWS:       if (value < 0 || value > UPD_TR_MAX || value % 8) return -1; break;
    case SPX_OPT_FUSE_DEPTH:       if (value < 0 || (value > 8 && value != fuse_max())) return -1; break;   // whole groups above 8
    case SPX_OPT_FUSE_MIN_BLOCKS:  if (value < 0 || value > 4) return -1; break;
    case SPX_OPT_FUSE_PRICING:     if (value < 0 || value > 2) return -1; break;
    case SPX_OPT_FUSE_LOOKAHEAD:   if (value < 0 || value > 2) return -1; break;
    case SPX_OPT_FUSE_TILE_ROWS:   if (value < 0 || value > 4096 || value % 8) return -1; break;
    case SPX_OPT_FUSE_PAIRS:       if (value < 0 || value > 2) return -1; break;
    case SPX_OPT_SHARD_THREADS:    if (value < 0 || value > 512 || value % 32 || value == 32) return -1; break;
    case SPX_OPT_SHARD_CTAS:       if (value < 0 || value > 4096) return -1; break;
    case SPX_OPT_CLUSTER_SIZE:     if (value < 0 || value > 16 || (value & (value - 1))) return -1; break;
    default: return -1;
    }
    g_opt[key] = value;
    return 0;
}

cudaError_t update(const double *Ain, double *Aout, const double *bin, double *bout, int n,
                   int m_loc, int64_t ld, int64_t col0, spx_state *st, const double *colbuf,
                   int32_t *rowlab, int32_t *collab, int32_t *trace, int ahead, cudaStream_t stream) {
    const int tr = pick_tr(n, m_loc);
    dim3 grid((unsigned)((m_loc + UPD_TC - 1) / UPD_TC), (unsigned)((n + 1 + tr - 1) / tr));
    if (grid.x == 0) grid.x = 1;      // a shard with no columns still updates b
#define SPX_LAUNCH_TILED(MINB)                                                                      \
    update_tiled_kernel<MINB><<<grid, UPD_THREADS, 0, stream>>>(Ain, Aout, bin, bout, n, m_loc, ld, \
                                                               col0, tr, ahead, st, colbuf, rowlab, collab, trace)
    switch ((int)g_opt[SPX_OPT_TILED_MIN_BLOCKS]) {
    case 1: SPX_LAUNCH_TILED(1); break;
    case 2: SPX_LAUNCH_TILED(2); break;
    case 3: SPX_LAUNCH_TILED(3); break;
    default: SPX_LAUNCH_TILED(4); break;
    }
#undef SPX_LAUNCH_TILED
    spx_host::count_launch();
    return cudaGetLastError();
}

cudaError_t selftest_division(const double *a, const double *p, int64_t count, int64_t np,
                              unsigned long long *d_mismatches, double *d_first_bad, cudaStream_t stream) {
    division_selftest_kernel<<<sm_count() * 8, 256, 0, stream>>>(a, p, count, np, d_mismatches, d_first_bad);
    spx_host::count_launch();
    return cudaGetLastError();
}

cudaError_t extract(const double *b, int n, int m, const int32_t *collab, const double *function,
                    double *x, double *obj, cudaStream_t stream) {
    cudaError_t e = cudaMemsetAsync(x, 0, (size_t)m * sizeof(double), stream);
    if (e != cudaSuccess) return e;
    const int blocks = max(1, min(1024, (n + 255) / 256));
    extract_kernel<<<blocks, 256, 0, stream>>>(b, n, m, collab, function, x, obj);
    objective_kernel<<<1, 32, 0, stream>>>(m, function, x, obj);
    spx_host::count_launch(2);
    return cudaGetLastError();
}

cudaError_t init_state(spx_state *st, int32_t *rowlab, int32_t *collab, int n, int m,
                       int64_t max_pivots, cudaStream_t stream) {
    const int blocks = max(1, min(1024, (max(n, m) + 255) / 256));
    init_state_kernel<<<blocks, 256, 0, stream>>>(st, rowlab, collab, n, m, max_pivots);
    spx_host::count_launch();
    return cudaGetLastError();
}

} // namespace spx_launch
