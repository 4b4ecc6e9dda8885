// spx_cluster.cu — K7: whole-LP solver for batches of mid-size LPs, one thread-block CLUSTER per LP: the loop of
// get_solution(), /root/reference/src/simplex.py:179-199, with pick_element() (:70-141) and recalculate_matrix()
// (:143-177) inlined, as in K4 (spx_batched.cu), for tables too big for one CTA's shared memory.
//
// Layout.  CTA k of a cluster of S owns the body rows [k*R, k*R + R) (R = ceil(n/S)), each row [a_1..a_m, b] as in
// the reference-flat table, so a band is one contiguous slice of the LP's d_T slice.  The f row is REPLICATED: every
// CTA applies the same operations to its copy, so the copies stay bit-identical and every CTA finds the entering
// column of the f row on its own.  The header labels rl (one per column) are spread over the CTAs in slices of
// Q = ceil(m/S); the row labels cl live with their rows.
//
// Update in place.  A new cell depends only on the old cell, the OLD pivot row, the OLD pivot-column entry of its row
// and p (:156,:160,:163,:173-175), so each CTA keeps two stashes instead of K4's second table: the pivot row, pulled
// from its owner over distributed shared memory, and the band's pivot-column entries.  Per CTA, in bytes:
//     8 * (R*(m+1) + m + (m+1) + R)  +  4 * (R + Q)        band, f row, pivot row, pivot column; cl, rl slice
// which must fit CLUSTER_DYN_BYTES (227 KB minus the static reduction scratch).
//
// One pivot, per CTA:
//   pricing   the entering column c_f of the (replicated) f row; one pass over the band folds the first row with
//             b < 0 (and the first positive cell of that row) and the ratio scan of column c_f into a partial, which
//             the CTA publishes in its own shared memory;
//   barrier A cluster.sync();
//   decision  warp 0 of EVERY CTA merges the S partials (first-index minima, ratio_merge: order independent), so all
//             CTAs reach the same (status, r, c) without another round; the phase-1 row's first positive cell comes
//             from the partial of the row's owner;
//   stash     pull the old pivot row from its owner, copy the band's pivot-column entries; swap the two labels
//             (read the peer's old label now, write after the barrier);
//   barrier B cluster.sync(): nobody overwrites a band before every CTA holds the old pivot row.  It also keeps the
//             partials of pivot k+1 (written after B) from overwriting those of pivot k (read before B);
//   update    the band and the f row in place, one division by the pivot (pivot_div, reciprocal hoisted).
// A final cluster.sync() keeps every CTA's shared memory alive until no peer can read it any more.
#include "spx_cluster.cuh"

namespace cg = cooperative_groups;

namespace {

using namespace spx;

// The body of both kernels.  RAGGED == false: shape, R, Q and offsets from the arguments (one shape per launch).
// RAGGED == true: LP order[blockIdx.x / S] of a ragged batch, its shape and offsets from lps[], R and Q from its shape.
// WARM == true: a resume (spx_warm_solve_*): each CTA reads the labels of its band and of its header slice from
// a.rowlab / a.collab, f0 and f1 for obj come from `function` (packed as x) in the epilogue, and no label outside
// [0, m) indexes x or s_x01.
template <bool RAGGED, bool WARM>
__device__ __forceinline__ void cluster_body(const ClusterArgs &a, const RaggedLp *__restrict__ lps,
                                             const int32_t *__restrict__ order, const double *function) {
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ Scratch sc;
    __shared__ Partial s_part;
    __shared__ int s_ctl[3];                               // {status, r, c} of the merged decision
    __shared__ double s_x01[2];                            // rank 0: b of the rows labelled x1, x2 (:49)

    RaggedLp d;
    if (RAGGED) d = lps[order[blockIdx.x / (unsigned)a.S]];
    const int n = RAGGED ? d.n : a.n, m = RAGGED ? d.m : a.m, w1 = m + 1, S = a.S;
    const int R = RAGGED ? (n + S - 1) / S : a.R, Q = RAGGED ? (m + S - 1) / S : a.Q;
    const int rank = (int)cluster.block_rank();
    const int64_t lp = RAGGED ? (int64_t)order[blockIdx.x / (unsigned)S] : (int64_t)(blockIdx.x / (unsigned)S);
    const int tid = (int)threadIdx.x, nt = (int)blockDim.x;
    const int r0 = rank * R;                               // first body row of this band
    const int rows = max(0, min(R, n - r0));
    const int j0 = rank * Q;                               // first column of this CTA's header-label slice
    const int cols = max(0, min(Q, m - j0));
    const int bandcells = rows * w1;

    double *band = reinterpret_cast<double *>(smem_raw);   // [R][w1]
    double *f    = band + (size_t)R * w1;                  // [m]  replicated f row
    double *prow = f + m;                                  // [w1] stash: old pivot row
    double *pcol = prow + w1;                              // [R]  stash: old pivot-column entries of the band
    int32_t *cl  = reinterpret_cast<int32_t *>(pcol + R);  // [R]  labels of the band's rows ('y1'..'yn' :31)
    int32_t *rl  = cl + R;                                 // [Q]  header labels of columns j0.. ('x1'..'xm' :30)

    const int64_t cells = (int64_t)n * w1 + m;
    const int fo = n * w1;                                 // offset of the f row
    double *Tg = a.T + (RAGGED ? d.t : lp * cells);
    for (int k = tid; k < bandcells; k += nt) band[k] = Tg[(int64_t)r0 * w1 + k];
    for (int j = tid; j < m; j += nt) f[j] = Tg[fo + j];
    if constexpr (WARM) {
        for (int i = tid; i < rows; i += nt) cl[i] = a.collab[(RAGGED ? d.xn : lp * n) + r0 + i];
        for (int j = tid; j < cols; j += nt) rl[j] = a.rowlab[(RAGGED ? d.xm : lp * m) + j0 + j];
    } else {
        for (int i = tid; i < rows; i += nt) cl[i] = m + r0 + i;
        for (int j = tid; j < cols; j += nt) rl[j] = j0 + j;
    }
    if (tid < 2) s_x01[tid] = 0.0;
    cluster.sync();                                        // every CTA runs and is loaded before any DSMEM access
    const double f0 = (m >= 1) ? f[0] : 0.0;               // self.function is never mutated (:29,:49)
    const double f1 = (m >= 2) ? f[1] : 0.0;
    const float inv_w1 = 1.0f / (float)w1;

    int npiv = 0, status;
    double *snap = a.snap ? a.snap + (RAGGED ? d.sn : lp * (int64_t)(a.max_pivots + 1) * cells) : nullptr;
    int32_t *trace = a.trace ? a.trace + (RAGGED ? 2 * d.tr : lp * (int64_t)a.max_pivots * 2) : nullptr;

    for (;;) {
        if (snap) {
            double *sg = snap + (int64_t)npiv * cells;
            for (int k = tid; k < bandcells; k += nt) sg[(int64_t)r0 * w1 + k] = band[k];
            if (rank == 0) for (int j = tid; j < m; j += nt) sg[fo + j] = f[j];
        }
        // ---- K1: entering column of the f row (:94-98), the same in every CTA
        const int cf = f_row_entering(f, m, a.rule, sc);
        // ---- one pass over the band: phase-1 row (:72-76) and the ratio scan of column cf (:107-136)
        Ratio q = ratio_identity();
        int key = SPX_NONE, bneg = SPX_NONE;
        for (int i = tid; i < rows; i += nt) {
            const double b_i = band[i * w1 + m];
            if (b_i < 0.0) bneg = min(bneg, i);
            if (cf != SPX_NONE) {
                const bool first = (q.elig_row == SPX_NONE);
                const bool is_nan = ratio_accumulate(q, r0 + i, band[i * w1 + cf], b_i);
                if (first && q.elig_row != SPX_NONE) key = 2 * (r0 + i) + (is_nan ? 1 : 0);
            }
        }
        block_min_int2(bneg, key, sc);
        if (cf != SPX_NONE) q = block_ratio_reduce(q, sc);
        int bcol = SPX_NONE;                               // first positive cell of the phase-1 row (:81-85)
        if (bneg != SPX_NONE) bcol = block_first_index(band + bneg * w1, m, IsPos(), sc);
        if (tid == 0) {
            s_part.q = q;
            s_part.elig_key = key;
            s_part.bneg_row = (bneg == SPX_NONE) ? SPX_NONE : r0 + bneg;
            s_part.bneg_col = bcol;
        }
        cluster.sync();                                    // A: every partial is published

        // ---- decision: each CTA merges the S partials itself
        if (tid < 32) cluster_decide(cluster, &s_part, S, cf, s_ctl);
        __syncthreads();
        status = s_ctl[0];
        const int r = s_ctl[1], c = s_ctl[2];
        if (status != SPX_PIVOT) break;
        if (npiv >= (RAGGED ? d.max_pivots : a.max_pivots)) { status = SPX_CAP; break; }

        // ---- stash the old pivot row (from its owner) and the band's old pivot-column entries
        const int owner = r / R, holder = c / Q;           // owners of row r and of the header label of column c
        const double *orow = cluster.map_shared_rank(band, owner) + (size_t)(r - owner * R) * w1;
        for (int j = tid; j < w1; j += nt) prow[j] = orow[j];
        for (int i = tid; i < rows; i += nt) pcol[i] = band[i * w1 + c];
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
        for (int k = tid; k < bandcells; k += nt) {
            int i = __float2int_rz((float)k * inv_w1), j = k - i * w1;     // k < 2^24: off by at most one row
            if (j < 0) { --i; j += w1; } else if (j >= w1) { ++i; j -= w1; }
            const double t = band[k];
            const double ci = pcol[i];
            const bool pr = (r0 + i == r), pc = (j == c);
            double num = __dsub_rn(__dmul_rn(t, p), __dmul_rn(prow[j], ci));
            num = pc ? ci : num;
            num = pr ? -t : num;
            num = (pr && pc) ? 1.0 : num;
            band[k] = pivot_div(num, d);
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

    // ---- epilogue: final table, labels, find_optimum()/f() (:48-68)
    for (int k = tid; k < bandcells; k += nt) Tg[(int64_t)r0 * w1 + k] = band[k];
    if (rank == 0) for (int j = tid; j < m; j += nt) Tg[fo + j] = f[j];
    double *xg = a.x ? a.x + (RAGGED ? d.xm : lp * m) : nullptr;
    // labels are a permutation of 0..n+m-1: x_j is the b of the row labelled x_j, or 0 when a column carries it
    for (int i = tid; i < rows; i += nt) {
        const int lab = cl[i];
        if ((!WARM || lab >= 0) && lab < m) {
            const double v = band[i * w1 + m];
            if (xg) xg[lab] = v;
            if (lab < 2) *cluster.map_shared_rank(&s_x01[lab], 0) = v;
        }
        if (a.collab) a.collab[(RAGGED ? d.xn : lp * n) + r0 + i] = lab;
    }
    for (int j = tid; j < cols; j += nt) {
        const int lab = rl[j];
        if (xg && (!WARM || lab >= 0) && lab < m) xg[lab] = 0.0;
        if (a.rowlab) a.rowlab[(RAGGED ? d.xm : lp * m) + j0 + j] = lab;
    }
    cluster.sync();                                        // s_x01 complete; no CTA leaves while a peer may read it
    if (rank == 0 && tid == 0) {
        a.status[lp] = status;
        a.npiv[lp] = npiv;
        if (a.obj) {
            const double *fn = function + (RAGGED ? d.xm : lp * m);
            const double g0 = WARM ? fn[0] : f0, g1 = WARM && m >= 2 ? fn[1] : f1;
            a.obj[lp] = (m >= 2) ? __dadd_rn(__dmul_rn(g0, s_x01[0]), __dmul_rn(g1, s_x01[1])) : 0.0;
        }
    }
}

__global__ void __launch_bounds__(CLUSTER_THREADS, 1) cluster_kernel(ClusterArgs a) {
    cluster_body<false, false>(a, nullptr, nullptr, nullptr);
}

// a ragged batch: the LPs order[0 .. a.B) of one cluster size a.S, each cluster its own shape (a.n, a.m, a.R, a.Q unused)
__global__ void __launch_bounds__(CLUSTER_THREADS, 1)
ragged_cluster_kernel(ClusterArgs a, const RaggedLp *__restrict__ lps, const int32_t *__restrict__ order) {
    cluster_body<true, false>(a, lps, order, nullptr);
}

// the resumes of the two kernels above (spx_warm_solve_*): function [B][m] or packed as x, null without obj
__global__ void __launch_bounds__(CLUSTER_THREADS, 1) cluster_warm_kernel(ClusterArgs a, const double *function) {
    cluster_body<false, true>(a, nullptr, nullptr, function);
}

__global__ void __launch_bounds__(CLUSTER_THREADS, 1)
ragged_cluster_warm_kernel(ClusterArgs a, const RaggedLp *__restrict__ lps, const int32_t *__restrict__ order,
                           const double *function) {
    cluster_body<true, true>(a, lps, order, function);
}

// the per-CTA footprint of the header comment, for S CTAs per LP
int64_t cluster_bytes(int64_t n, int64_t m, int S) {
    const int64_t R = (n + S - 1) / S, Q = (m + S - 1) / S;
    return 8 * (R * (m + 2) + 2 * m + 1) + 4 * (R + Q);
}

} // namespace

namespace spx_launch {

bool cluster_fits(int64_t n, int64_t m, int S) {
    return n >= 1 && m >= 1 && cluster_bytes(n, m, S) <= (int64_t)CLUSTER_DYN_BYTES;
}

// smallest S in {1, 2, 4, 8, 16} whose footprint fits, 0 when none does
int cluster_size(int64_t n, int64_t m) {
    for (int S = 1; S <= CLUSTER_MAX_S; S *= 2)
        if (cluster_fits(n, m, S)) return S;
    return 0;
}

// S CTAs per LP (validated by the caller); returns cudaErrorInvalidClusterSize when the device cannot co-schedule
// one cluster of this size and footprint
cudaError_t solve_batched_cluster(int64_t B, int n, int m, int S, int max_pivots, const BatchIO &io,
                                  cudaStream_t stream) {
    const ClusterArgs a = cluster_args(io, B, n, m, S, max_pivots);
    if (io.warm) return launch_cluster_kernel<cluster_warm_kernel>(S, B, cluster_bytes(n, m, S), stream, a, io.function);
    return launch_cluster_kernel<cluster_kernel>(S, B, cluster_bytes(n, m, S), stream, a);
}

int64_t ragged_cluster_bytes(int n, int m, int S) { return cluster_bytes(n, m, S); }

// one launch of a ragged plan: the l.count LPs order[l.first ..] at cluster size l.S, l.smem = the largest footprint
// among them; cudaErrorInvalidClusterSize when the device cannot co-schedule one such cluster
cudaError_t solve_ragged_cluster(const PlanView &v, const RaggedLaunch &l, const BatchIO &io, cudaStream_t stream) {
    const ClusterArgs a = cluster_args(io, l.count, 0, 0, l.S, 0);
    const int32_t *order = v.d_order + l.first;
    if (io.warm)
        return launch_cluster_kernel<ragged_cluster_warm_kernel>(l.S, l.count, l.smem, stream, a, v.d_lps, order,
                                                                 io.function);
    return launch_cluster_kernel<ragged_cluster_kernel>(l.S, l.count, l.smem, stream, a, v.d_lps, order);
}

} // namespace spx_launch
