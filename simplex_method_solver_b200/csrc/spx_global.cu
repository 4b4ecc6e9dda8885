// spx_global.cu — K8: whole-LP solver for batches of LPs too large for one cluster's shared memory, one
// thread-block CLUSTER per LP with the table in GLOBAL memory: the loop of get_solution(),
// /root/reference/src/simplex.py:179-199, with pick_element() (:70-141) and recalculate_matrix() (:143-177) inlined,
// as in K7 (spx_cluster.cu), whose protocol it keeps.
//
// Layout.  CTA k of a cluster of S owns the body rows [k*R, k*R + R) (R = ceil(n/S)), each row [a_1..a_m, b] as in
// the reference-flat table, so a band is one contiguous slice of the LP's d_T slice; it is updated IN PLACE in d_T.
// Shared memory holds only what every pivot reads many times: the replicated f row, the old-pivot-row stash, the
// band's old pivot-column entries, the band's row labels cl and a slice of Q = ceil(m/S) header labels rl.  Per CTA,
// in bytes:
//     8 * (m + (m+1) + R)  +  4 * (R + Q)                f row, pivot row, pivot column; cl, rl slice
// which must fit CLUSTER_DYN_BYTES (227 KB minus the static reduction scratch): m <= 11,519 at S = 1 and 14,177 at
// S = 16; at m = 2,000, n <= 15,866 at S = 1 and 263,856 at S = 16.
//
// One pivot, per CTA (K7's protocol):
//   pricing   the entering column c_f of the (replicated) f row; one pass over the band's rows folds the first row
//             with b < 0 (and the first positive cell of that row) and the ratio scan of column c_f into a partial,
//             published in the CTA's shared memory;
//   barrier A cluster.sync();
//   decision  warp 0 of EVERY CTA merges the S partials (cluster_decide), so all CTAs reach the same (status, r, c);
//   stash     the old pivot row r from global memory, the band's old pivot-column entries; the two labels (read the
//             peer's old label now over DSMEM, write after B);
//   barrier B cluster.sync(): no CTA overwrites its band before every CTA holds the old pivot row;
//   update    the band (16-byte loads and stores, several in flight per thread) and the f row in place, one
//             division by the pivot (pivot_div, reciprocal hoisted).
// A final cluster.sync() keeps every CTA's shared memory alive until no peer can read it any more.
//
// Memory ordering.  d_T is read and written by this kernel, so every read of it goes through ld_l2 / ld_l2_v2
// (ld.global.cg: from L2, never the non-coherent path or a stale L1 line).  A CTA reads cells another CTA wrote only
// in one place, the pivot row (owned by one CTA, read by all); the owner wrote it in the update of the previous
// pivot, before its arrival at barrier A, whose release/acquire at cluster scope orders it before the read.  Every
// other read of d_T is of the CTA's own band, ordered by __syncthreads().
#include "spx_cluster.cuh"

namespace cg = cooperative_groups;

namespace {

using namespace spx;

// one CTA of 512 threads per SM: the pricing and the division's slow path need more than the 64 registers two would
// leave (spills); six 16-byte loads in flight per thread keep 48 KB per SM in flight for the update
constexpr int    GLOBAL_MIN_CTAS  = 1;
constexpr int    GLOBAL_UNROLL    = 6;

__device__ __forceinline__ double ld_l2(const double *p) {
    double v;
    asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double2 ld_l2_v2(const double *p) {
    double2 v;
    asm volatile("ld.global.cg.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}

// The body of both kernels.  RAGGED == false: shape, R, Q and offsets from the arguments (one shape per launch).
// RAGGED == true: LP order[blockIdx.x / S] of a ragged batch, its shape and offsets from lps[], R and Q from its shape
// (as cluster_body in spx_cluster.cu).  WARM == true: a resume, as cluster_body's.
template <bool RAGGED, bool WARM>
__device__ __forceinline__ void global_body(const ClusterArgs &a, const RaggedLp *__restrict__ lps,
                                            const int32_t *__restrict__ order, const double *function) {
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ Scratch sc;
    __shared__ Partial s_part;
    __shared__ int s_ctl[3];                               // {status, r, c} of the merged decision
    __shared__ double s_x01[2];                            // rank 0: b of the rows labelled x1, x2 (:49)

    RaggedLp lpd;
    if (RAGGED) lpd = lps[order[blockIdx.x / (unsigned)a.S]];
    const int n = RAGGED ? lpd.n : a.n, m = RAGGED ? lpd.m : a.m, w1 = m + 1, S = a.S;
    const int R = RAGGED ? (n + S - 1) / S : a.R, Q = RAGGED ? (m + S - 1) / S : a.Q;
    const int rank = (int)cluster.block_rank();
    const int64_t lp = RAGGED ? (int64_t)order[blockIdx.x / (unsigned)S] : (int64_t)(blockIdx.x / (unsigned)S);
    const int tid = (int)threadIdx.x, nt = (int)blockDim.x;
    const int r0 = rank * R;                               // first body row of this band
    const int rows = max(0, min(R, n - r0));
    const int j0 = rank * Q;                               // first column of this CTA's header-label slice
    const int cols = max(0, min(Q, m - j0));
    const int64_t bandcells = (int64_t)rows * w1;

    double *f    = reinterpret_cast<double *>(smem_raw);   // [m]  replicated f row
    double *prow = f + m;                                  // [w1] stash: old pivot row
    double *pcol = prow + w1;                              // [R]  stash: old pivot-column entries of the band
    int32_t *cl  = reinterpret_cast<int32_t *>(pcol + R);  // [R]  labels of the band's rows ('y1'..'yn' :31)
    int32_t *rl  = cl + R;                                 // [Q]  header labels of columns j0.. ('x1'..'xm' :30)

    const int64_t cells = (int64_t)n * w1 + m;
    const int64_t fo = (int64_t)n * w1;                    // offset of the f row
    double *Tg = a.T + (RAGGED ? lpd.t : lp * cells);
    double *band = Tg + (int64_t)r0 * w1;                  // [rows][w1], in place
    // 16-byte accesses: a band starts at 8-byte alignment only, so a misaligned first cell and an odd last cell
    // are done one at a time
    const int head = (bandcells > 0 && (reinterpret_cast<uintptr_t>(band) & 15)) ? 1 : 0;
    const int64_t pairs = (bandcells - head) >> 1;
    const bool tail = bandcells > head && ((bandcells - head) & 1);
    const double inv_w1 = 1.0 / (double)w1;

    for (int j = tid; j < m; j += nt) f[j] = ld_l2(Tg + fo + j);
    if constexpr (WARM) {
        for (int i = tid; i < rows; i += nt) cl[i] = a.collab[(RAGGED ? lpd.xn : lp * n) + r0 + i];
        for (int j = tid; j < cols; j += nt) rl[j] = a.rowlab[(RAGGED ? lpd.xm : lp * m) + j0 + j];
    } else {
        for (int i = tid; i < rows; i += nt) cl[i] = m + r0 + i;
        for (int j = tid; j < cols; j += nt) rl[j] = j0 + j;
    }
    if (tid < 2) s_x01[tid] = 0.0;
    cluster.sync();                                        // every CTA runs and is loaded before any DSMEM access
    const double f0 = (m >= 1) ? f[0] : 0.0;               // self.function is never mutated (:29,:49)
    const double f1 = (m >= 2) ? f[1] : 0.0;

    int npiv = 0, status;
    double *snap = a.snap ? a.snap + (RAGGED ? lpd.sn : lp * (int64_t)(a.max_pivots + 1) * cells) : nullptr;
    int32_t *trace = a.trace ? a.trace + (RAGGED ? 2 * lpd.tr : lp * (int64_t)a.max_pivots * 2) : nullptr;

    for (;;) {
        if (snap) {
            double *sg = snap + (int64_t)npiv * cells;
            for (int64_t k = tid; k < bandcells; k += nt) sg[(int64_t)r0 * w1 + k] = ld_l2(band + k);
            if (rank == 0) for (int j = tid; j < m; j += nt) sg[fo + j] = f[j];
        }
        // ---- K1: entering column of the f row (:94-98), the same in every CTA
        const int cf = f_row_entering(f, m, a.rule, sc);
        // ---- one pass over the band's rows: phase-1 row (:72-76) and the ratio scan of column cf (:107-136)
        Ratio q = ratio_identity();
        int key = SPX_NONE, bneg = SPX_NONE;
        for (int i = tid; i < rows; i += nt) {
            const double *row = band + (int64_t)i * w1;
            const double b_i = ld_l2(row + m);
            if (b_i < 0.0) bneg = min(bneg, i);
            if (cf != SPX_NONE) {
                const bool first = (q.elig_row == SPX_NONE);
                const bool is_nan = ratio_accumulate(q, r0 + i, ld_l2(row + cf), b_i);
                if (first && q.elig_row != SPX_NONE) key = 2 * (r0 + i) + (is_nan ? 1 : 0);
            }
        }
        block_min_int2(bneg, key, sc);
        if (cf != SPX_NONE) q = block_ratio_reduce(q, sc);
        int bcol = SPX_NONE;                               // first positive cell of the phase-1 row (:81-85)
        if (bneg != SPX_NONE) {
            const double *row = band + (int64_t)bneg * w1;
            bcol = block_first_index_fn(m, [row](int j) { return ld_l2(row + j); }, IsPos(), sc);
        }
        if (tid == 0) {
            s_part.q = q;
            s_part.elig_key = key;
            s_part.bneg_row = (bneg == SPX_NONE) ? SPX_NONE : r0 + bneg;
            s_part.bneg_col = bcol;
        }
        cluster.sync();                                    // A: every partial is published; the pivot row is final

        // ---- decision: each CTA merges the S partials itself
        if (tid < 32) cluster_decide(cluster, &s_part, S, cf, s_ctl);
        __syncthreads();
        status = s_ctl[0];
        const int r = s_ctl[1], c = s_ctl[2];
        if (status != SPX_PIVOT) break;
        if (npiv >= (RAGGED ? lpd.max_pivots : a.max_pivots)) { status = SPX_CAP; break; }

        // ---- stash the old pivot row and the band's old pivot-column entries
        const int owner = r / R, holder = c / Q;           // owners of row r and of the header label of column c
        // row r was written by its owner before barrier A (the update of the previous pivot): read from L2
        const double *orow = Tg + (int64_t)r * w1;
        for (int j = tid; j < w1; j += nt) prow[j] = ld_l2(orow + j);
        for (int i = tid; i < rows; i += nt) pcol[i] = ld_l2(band + (int64_t)i * w1 + c);
        const double fc = f[c];
        int32_t lab_r = 0, lab_c = 0;                      // :152, old labels read before B, written after B
        if (tid == 0) {
            if (rank == holder) lab_r = *cluster.map_shared_rank(cl + (r - owner * R), owner);
            if (rank == owner) lab_c = *cluster.map_shared_rank(rl + (c - holder * Q), holder);
            if (trace && rank == 0) { trace[2 * npiv] = r; trace[2 * npiv + 1] = c; }
        }
        cluster.sync();                                    // B: every CTA holds the old pivot row

        // ---- K3 in place (:149-177): the four cell kinds (:156 pivot row, :160 pivot column, :163 pivot cell,
        // :173-175 the rest) differ only in the numerator, so one division by the pivot serves them all
        const double p = prow[c];
        const PivotDiv d = pivot_div_prepare(p);
        const int rloc = r - r0;                           // the pivot row in band coordinates (may be outside)
        auto cell = [&](double t, int i, int j) {
            const double ci = pcol[i];
            const bool pr = (i == rloc), pc = (j == c);
            double num = __dsub_rn(__dmul_rn(t, p), __dmul_rn(prow[j], ci));
            num = pc ? ci : num;
            num = pr ? -t : num;
            num = (pr && pc) ? 1.0 : num;
            return pivot_div(num, d);
        };
        // (row, column) of band cell k, exact: the double quotient is off by at most one row for any band size
        auto locate = [&](int64_t k, int &i, int &j) {
            i = (int)((double)k * inv_w1);
            int64_t jj = k - (int64_t)i * w1;
            if (jj < 0) { --i; jj += w1; } else if (jj >= w1) { ++i; jj -= w1; }
            j = (int)jj;
        };
        if (head && tid == 0) band[0] = cell(ld_l2(band), 0, 0);
        if (tail && tid == nt - 1) {
            int i, j;
            locate(bandcells - 1, i, j);
            band[bandcells - 1] = cell(ld_l2(band + bandcells - 1), i, j);
        }
        double *vb = band + head;                          // 16-byte aligned
        for (int64_t v0 = tid; v0 < pairs; v0 += (int64_t)nt * GLOBAL_UNROLL) {
            double2 t[GLOBAL_UNROLL];
#pragma unroll
            for (int u = 0; u < GLOBAL_UNROLL; ++u) {
                const int64_t v = v0 + (int64_t)u * nt;
                if (v < pairs) t[u] = ld_l2_v2(vb + 2 * v);
            }
#pragma unroll
            for (int u = 0; u < GLOBAL_UNROLL; ++u) {
                const int64_t v = v0 + (int64_t)u * nt;
                if (v < pairs) {
                    int i, j;
                    locate(head + 2 * v, i, j);
                    double2 o;
                    o.x = cell(t[u].x, i, j);
                    if (++j == w1) { j = 0; ++i; }
                    o.y = cell(t[u].y, i, j);
                    *reinterpret_cast<double2 *>(vb + 2 * v) = o;
                }
            }
        }
        for (int j = tid; j < m; j += nt) {
            const double t = f[j];
            double num = __dsub_rn(__dmul_rn(t, p), __dmul_rn(prow[j], fc));
            num = (j == c) ? fc : num;
            f[j] = pivot_div(num, d);
        }
        if (tid == 0) {
            if (rank == holder) rl[c - j0] = lab_r;
            if (rank == owner) cl[r - r0] = lab_c;
        }
        __syncthreads();
        ++npiv;
    }

    // ---- epilogue: the band is final in place; f row, labels, find_optimum()/f() (:48-68)
    if (rank == 0) for (int j = tid; j < m; j += nt) Tg[fo + j] = f[j];
    double *xg = a.x ? a.x + (RAGGED ? lpd.xm : lp * m) : nullptr;
    // labels are a permutation of 0..n+m-1: x_j is the b of the row labelled x_j, or 0 when a column carries it
    for (int i = tid; i < rows; i += nt) {
        const int lab = cl[i];
        if ((!WARM || lab >= 0) && lab < m) {
            const double v = ld_l2(band + (int64_t)i * w1 + m);
            if (xg) xg[lab] = v;
            if (lab < 2) *cluster.map_shared_rank(&s_x01[lab], 0) = v;
        }
        if (a.collab) a.collab[(RAGGED ? lpd.xn : lp * n) + r0 + i] = lab;
    }
    for (int j = tid; j < cols; j += nt) {
        const int lab = rl[j];
        if (xg && (!WARM || lab >= 0) && lab < m) xg[lab] = 0.0;
        if (a.rowlab) a.rowlab[(RAGGED ? lpd.xm : lp * m) + j0 + j] = lab;
    }
    cluster.sync();                                        // s_x01 complete; no CTA leaves while a peer may read it
    if (rank == 0 && tid == 0) {
        a.status[lp] = status;
        a.npiv[lp] = npiv;
        if (a.obj) {
            const double *fn = function + (RAGGED ? lpd.xm : lp * m);
            const double g0 = WARM ? fn[0] : f0, g1 = WARM && m >= 2 ? fn[1] : f1;
            a.obj[lp] = (m >= 2) ? __dadd_rn(__dmul_rn(g0, s_x01[0]), __dmul_rn(g1, s_x01[1])) : 0.0;
        }
    }
}

__global__ void __launch_bounds__(CLUSTER_THREADS, GLOBAL_MIN_CTAS) global_kernel(ClusterArgs a) {
    global_body<false, false>(a, nullptr, nullptr, nullptr);
}

// a ragged batch: the LPs order[0 .. a.B) at one cluster size a.S, each cluster its own shape (a.n, a.m, a.R, a.Q,
// a.max_pivots unused)
__global__ void __launch_bounds__(CLUSTER_THREADS, GLOBAL_MIN_CTAS)
ragged_global_kernel(ClusterArgs a, const RaggedLp *__restrict__ lps, const int32_t *__restrict__ order) {
    global_body<true, false>(a, lps, order, nullptr);
}

// the resumes of the two kernels above (spx_warm_solve_*): function [B][m] or packed as x, null without obj
__global__ void __launch_bounds__(CLUSTER_THREADS, GLOBAL_MIN_CTAS) global_warm_kernel(ClusterArgs a, const double *function) {
    global_body<false, true>(a, nullptr, nullptr, function);
}

__global__ void __launch_bounds__(CLUSTER_THREADS, GLOBAL_MIN_CTAS)
ragged_global_warm_kernel(ClusterArgs a, const RaggedLp *__restrict__ lps, const int32_t *__restrict__ order,
                          const double *function) {
    global_body<true, true>(a, lps, order, function);
}

// the per-CTA footprint of the header comment, for S CTAs per LP
int64_t global_bytes(int64_t n, int64_t m, int S) {
    const int64_t R = (n + S - 1) / S, Q = (m + S - 1) / S;
    return 8 * (2 * m + 1 + R) + 4 * (R + Q);
}

// The default cluster size of a K8 launch of `count` LPs on the current device: the S >= s_lo that keeps the most SMs
// busy, min(count, co-resident clusters at S) * S, the smaller S on ties; bytes(S) is the launch's footprint at S
// (which fits for every S >= s_lo: it does not grow with S).  A CTA streams its band at a rate bounded by its own
// bytes in flight, so an idle SM is lost bandwidth, while a larger S costs barrier time per pivot: a single LP gets
// 16 CTAs, a batch that fills the GPU at s_lo gets s_lo.
template <auto Kernel, typename Bytes>
cudaError_t busiest_cluster_size(int s_lo, int64_t count, Bytes bytes, int *S_out) {
    cudaError_t e = configure_cluster_kernel<Kernel>();
    if (e != cudaSuccess) return e;
    int64_t best = -1;
    for (int S = s_lo; S <= CLUSTER_MAX_S; S *= 2) {
        cudaLaunchAttribute attr[1];
        const cudaLaunchConfig_t cfg = cluster_launch_config(bytes(S), S, 1, attr, nullptr);
        int clusters = 0;
        e = cudaOccupancyMaxActiveClusters(&clusters, Kernel, &cfg);
        if (e != cudaSuccess) return e;
        const int64_t busy = (count < clusters ? count : (int64_t)clusters) * S;
        if (busy > best) { best = busy; *S_out = S; }
    }
    return cudaSuccess;
}

} // namespace

namespace spx_launch {

bool global_fits(int64_t n, int64_t m, int S) {
    return n >= 1 && m >= 1 && global_bytes(n, m, S) <= (int64_t)CLUSTER_DYN_BYTES;
}

// smallest S in {1, 2, 4, 8, 16} whose footprint fits, 0 when none does
int global_min_cluster_size(int64_t n, int64_t m) {
    for (int S = 1; S <= CLUSTER_MAX_S; S *= 2)
        if (global_fits(n, m, S)) return S;
    return 0;
}

// S for a solve of B LPs on the current device: SPX_OPT_CLUSTER_SIZE when set (0 if that S does not fit); else
// busiest_cluster_size() from S_min (0 when the LP does not fit)
cudaError_t global_cluster_size(int64_t n, int64_t m, int64_t B, int *S_out) {
    *S_out = 0;
    const int forced = (int)get_option(SPX_OPT_CLUSTER_SIZE);
    if (forced > 0) {
        *S_out = global_fits(n, m, forced) ? forced : 0;
        return cudaSuccess;
    }
    const int smin = global_min_cluster_size(n, m);
    if (smin == 0) return cudaSuccess;
    return busiest_cluster_size<global_kernel>(smin, B, [&](int S) { return global_bytes(n, m, S); }, S_out);
}

// S CTAs per LP (validated by the caller); returns cudaErrorInvalidClusterSize when the device cannot co-schedule
// one cluster of this size and footprint
cudaError_t solve_batched_global(int64_t B, int n, int m, int S, int max_pivots, const BatchIO &io,
                                 cudaStream_t stream) {
    const ClusterArgs a = cluster_args(io, B, n, m, S, max_pivots);
    if (io.warm) return launch_cluster_kernel<global_warm_kernel>(S, B, global_bytes(n, m, S), stream, a, io.function);
    return launch_cluster_kernel<global_kernel>(S, B, global_bytes(n, m, S), stream, a);
}

int64_t ragged_global_bytes(int n, int m, int S) { return global_bytes(n, m, S); }

// The S and footprint one K8 launch of a ragged plan runs at on the current device: as planned when l.pick_S == 0
// (no device needed), else busiest_cluster_size() from the planned S over the launch's largest footprint at each S
cudaError_t ragged_global_size(const PlanView &v, const RaggedLaunch &l, int *S_out, int64_t *smem_out) {
    // the largest footprint at S among the launch's LPs
    auto bytes = [&](int S) { return launch_max(v, l, [S](const RaggedLp &d) { return global_bytes(d.n, d.m, S); }); };
    *S_out = l.S;
    *smem_out = l.smem;
    if (!l.pick_S) return cudaSuccess;
    const cudaError_t e = busiest_cluster_size<ragged_global_kernel>(l.S, l.count, bytes, S_out);
    if (e != cudaSuccess) return e;
    *smem_out = bytes(*S_out);
    return cudaSuccess;
}

// one K8 launch of a ragged plan: the l.count LPs order[l.first ..] at S CTAs each with smem bytes per CTA (from
// ragged_global_size); cudaErrorInvalidClusterSize when the device cannot co-schedule one such cluster
cudaError_t solve_ragged_global(const PlanView &v, const RaggedLaunch &l, int S, int64_t smem, const BatchIO &io,
                                cudaStream_t stream) {
    const ClusterArgs a = cluster_args(io, l.count, 0, 0, S, 0);
    const int32_t *order = v.d_order + l.first;
    if (io.warm)
        return launch_cluster_kernel<ragged_global_warm_kernel>(S, l.count, smem, stream, a, v.d_lps, order,
                                                                io.function);
    return launch_cluster_kernel<ragged_global_kernel>(S, l.count, smem, stream, a, v.d_lps, order);
}

} // namespace spx_launch
