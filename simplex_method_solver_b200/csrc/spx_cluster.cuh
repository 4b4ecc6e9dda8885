// spx_cluster.cuh — what the two one-cluster-per-LP solvers, K7 (spx_cluster.cu, table in shared memory) and K8
// (spx_global.cu, table in global memory), share: the pricing steps (the entering column of the replicated f row and
// the merge of the S per-CTA partials into one pivot decision that every CTA reaches on its own), and the host launch.
#pragma once
#include <cooperative_groups.h>

#include "spx_block.cuh"
#include "spx_launch.cuh"

namespace spx {

constexpr int    CLUSTER_THREADS   = 512;
constexpr int    CLUSTER_MAX_S     = 16;
constexpr size_t CLUSTER_SMEM      = 227 * 1024;                    // shared memory of one CTA, static + dynamic
constexpr size_t CLUSTER_STATIC    = 2048;                          // reserved for the kernel's static scratch
constexpr size_t CLUSTER_DYN_BYTES = CLUSTER_SMEM - CLUSTER_STATIC;  // 230,400 bytes for the per-CTA footprint

// what one CTA knows about the pivot after folding its band
struct Partial {
    Ratio q;            // ratio scan of its rows for the f-row entering column (global row indices)
    int   elig_key;     // 2 * (its first eligible row) + (that row's ratio is NaN); SPX_NONE none
    int   bneg_row;     // its first row with b < 0 (global index); SPX_NONE none
    int   bneg_col;     // the first positive cell of that row; SPX_NONE none
};

struct EqKey {          // Dantzig: the f cell whose orderable image is the minimum
    unsigned long long key;
    __device__ bool operator()(double v) const { return v < 0.0 && orderable(v) == key; }
};

// a read of global memory another CTA of the cluster writes: from L2 (ld.global.cg), never a stale L1 line
__device__ __forceinline__ double ld_l2(const double *p) {
    double v;
    asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

// ---- devex (SPX_RULE_DEVEX) in a cluster: one copy of the weights per LP in its x slice wg[0..m), ONE PIVOT BEHIND.
// During the pricing of pivot k, wg holds w(k-1) (w(0) = 1 at pivot 0); every CTA prices with w(k) = w(k-1) updated by
// pivot k-1 on the fly, from its pivot-row stash (still pivot k-1's row) and w(k-1)[c(k-1)].  Between barriers A(k)
// and B(k), the owner of the header slice [j0, j0+Q) stores w(k) over w(k-1) there: every CTA has read w(k-1) before A
// (pricing), nobody reads wg again before B, and the store reads the stash before the CTA overwrites it with pivot
// k's row.  No barrier and no shared memory is added, and every CTA computes the same bits.
struct DevexPrev {
    int      c;     // column of the previous pivot, -1 before the first
    PivotDiv d;     // its pivot
    double   wc;    // w(k-1)[c], read in pricing k
};

// w(k)[j] from wg (= w(k-1)) and the previous pivot's row stash prow
__device__ __forceinline__ double devex_weight_now(const double *wg, const double *prow, const DevexPrev &pv, int j) {
    const double wj = ld_l2(wg + j);
    if (pv.c < 0) return wj;
    return devex_weight(wj, pivot_div(j == pv.c ? 1.0 : -prow[j], pv.d), pv.wc, j == pv.c);
}

// K1 under devex: the minimum of (devex_key, j) over the candidates f_j < 0, weight(j) = w_j; the whole CTA calls it
template <class Weight>
__device__ __forceinline__ int devex_entering(const double *f, int m, Weight weight, Scratch &sc) {
    unsigned long long best = ~0ull;
    int bj = SPX_NONE;
    for (int j = (int)threadIdx.x; j < m; j += (int)blockDim.x) {
        const double v = f[j];
        if (v < 0.0) {
            const unsigned long long k = devex_key(v, weight(j));
            if (k < best) { best = k; bj = j; }
        }
    }
    const unsigned long long g = block_min_u64(best, sc);
    return block_min_int(best == g ? bj : SPX_NONE, sc);
}

// K1: the entering column of the f row (:94-98), SPX_NONE when there is none; the whole CTA calls it
__device__ __forceinline__ int f_row_entering(const double *f, int m, int rule, Scratch &sc) {
    if (rule == SPX_RULE_REFERENCE) return block_first_index(f, m, IsNeg(), sc);
    unsigned long long best = ~0ull;                       // Dantzig: most negative, lowest index on ties
    for (int j = (int)threadIdx.x; j < m; j += (int)blockDim.x) {
        const double v = f[j];
        if (v < 0.0) { const unsigned long long k = orderable(v); best = k < best ? k : best; }
    }
    best = block_min_u64(best, sc);
    return (best == ~0ull) ? SPX_NONE : block_first_index(f, m, EqKey{best}, sc);
}

// The decision from the S partials (first-index minima, ratio_merge: order independent), so all CTAs of the
// cluster reach the same {status, r, c} without another round; the phase-1 row's first positive cell comes from
// the partial of the row's owner.  Warp 0 calls it after the barrier that publishes every partial; it writes ctl.
__device__ __forceinline__ void cluster_decide(cooperative_groups::cluster_group &cluster, Partial *part, int S,
                                               int cf, int *ctl) {
    const int tid = (int)threadIdx.x;
    Partial p;
    p.q = ratio_identity(); p.elig_key = SPX_NONE; p.bneg_row = SPX_NONE; p.bneg_col = SPX_NONE;
    if (tid < S) p = *cluster.map_shared_rank(part, tid);
    const int r1 = warp_min_int(p.bneg_row);
    const int c1 = warp_min_int(p.bneg_row == r1 ? p.bneg_col : SPX_NONE);
    int st, r = -1, c = -1;
    if (r1 != SPX_NONE) {                                  // phase 1
        if (c1 == SPX_NONE) st = SPX_INCORRECT;            // :88-89
        else { st = SPX_PIVOT; r = r1; c = c1; }           // :91
    } else if (cf == SPX_NONE) {
        st = SPX_OPTIMAL;                                  // :101-103
    } else {
        const Ratio g = warp_ratio_reduce(p.q);
        const int k2 = warp_min_int(p.elig_key);
        r = ratio_decide(g, k2 != SPX_NONE && (k2 & 1));
        st = (r < 0) ? SPX_NOCONV : SPX_PIVOT;             // :138-139
        c = cf;
    }
    if (tid == 0) { ctl[0] = st; ctl[1] = r; ctl[2] = c; }
}

// ---- Dantzig with Bland's rule on degenerate pivots (SPX_RULE_DANTZIG_BLAND) in a cluster ----
// The rule needs what today's one round (pricing, barrier A, decision) cannot give in two places: phase 1's entering
// column comes from row t, which only its owner holds and which is known only after the merge; and Bland's column needs
// the lowest header label, spread over the CTAs in slices of Q.  So the pick runs in ROUNDS, each one fold over every
// CTA's band into a DbPartial, a cluster barrier, and the same merge in every CTA:
//   round 1 (barrier A)  the first row with b < 0; phase 2's Dantzig column c_D (replicated f row) and its leaving
//                        row; phase 2's Bland column (each CTA over its header slice); the Dantzig column of each CTA's
//                        first row with b < 0 (phase 1's c_D when that row is t)
//   round 2 (barrier A2) phase 1: the leaving row of c_D, and Bland's column (each CTA over its slice of row t);
//                        phase 2, only after a degenerate step: the leaving row of Bland's column
//   round 3 (barrier A3) phase 1, only after a degenerate step: the leaving row of Bland's column
// so a pivot has, with barrier B, 2 barriers in phase 2, 3 in a degenerate step of phase 2 and in phase 1, and 4 in a
// degenerate step of phase 1.  Every choice is the minimum of a key (spx_common.cuh), so every S gives the same bits.
struct DbPartial {
    unsigned long long rk, sk;   // leaving row: the least (ratio key, row key) over the CTA's candidate rows; ~0 none
    unsigned long long bk;       // Bland: the least db_label_key over the CTA's candidate columns; ~0 none
    int dj;                      // round 1: the Dantzig column of the CTA's first row with b < 0; SPX_NONE none
    int bneg;                    // round 1: the CTA's first row with b < 0 (global index); SPX_NONE none
};

// the minima of N keys over the CTA, one barrier pair; the storage is the caller's (every warp finishes on its own)
template <int N>
__device__ __forceinline__ void block_min_keys(unsigned long long (&v)[N], unsigned long long (*red)[BLOCK_MAX_WARPS]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (int)(blockDim.x >> 5);
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] = warp_min_u64(v[k]);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < N; ++k) red[k][warp] = v[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] = warp_min_u64(lane < nw ? red[k][lane] : ~0ull);
    __syncthreads();                              // red may be reused right away
}

// One pick of SPX_RULE_DANTZIG_BLAND by every CTA of the cluster (the whole CTA calls it): returns SPX_PIVOT with
// (r, c), the same in every CTA, or the terminal status.  f: the replicated f row; the CTA's band is the rows
// [r0, r0 + rows) and its header slice the columns [j0, j0 + cols) with labels rl; cl: the band's row labels.
// own(i, j): cell j of band row i; row(t, j): cell j of body row t, owned by any CTA (read only between barriers A and
// B: its owner writes it only in the update, after B).
// Memory ordering: a partial is written by its CTA before its arrival at the round's barrier and read by its peers
// over DSMEM after it (release/acquire at cluster scope).  Rounds 1 and 3 write one partial and round 2 the other, so
// between a write of one and its next write lie two barriers: every peer has read it before the second.  Row t's cells
// were written by its owner in the update of the previous pivot, before barrier A of this one.
template <class Own, class Row>
__device__ __forceinline__ int cluster_db_pick(cooperative_groups::cluster_group &cluster, const double *f, int m, int S,
                                               int r0, int rows, int j0, int cols, const int32_t *rl,
                                               const int32_t *cl, Scratch &sc, Own own, Row row, int &r, int &c) {
    __shared__ DbPartial part[2];
    __shared__ unsigned long long red[2][BLOCK_MAX_WARPS];
    __shared__ int ctl[5];                                 // {status, r, c, column of the next round or -1, t}
    const int tid = (int)threadIdx.x, nt = (int)blockDim.x, lane = tid & 31;

    // ---- round 1
    const int cf = f_row_entering(f, m, SPX_RULE_DANTZIG, sc);   // phase 2's c_D
    unsigned long long k2[2] = {~0ull, ~0ull};                 // {ratio key, Bland key}
    unsigned long long sk = ~0ull;
    int bneg = SPX_NONE;
    for (int i = tid; i < rows; i += nt) {
        const double b = own(i, m);
        if (b < 0.0) bneg = min(bneg, i);
        if (cf != SPX_NONE) db_leave_fold(k2[0], sk, r0 + i, own(i, cf), b, SPX_NONE, cl[i]);
    }
    for (int j = tid; j < cols; j += nt)
        if (f[j0 + j] < 0.0) k2[1] = min(k2[1], db_label_key(rl[j], j0 + j));
    const unsigned long long mine = k2[0];
    block_min_keys<2>(k2, red);
    unsigned long long s2[2] = {mine == k2[0] ? sk : ~0ull, (unsigned long long)(unsigned)bneg};
    block_min_keys<2>(s2, red);
    bneg = (int)s2[1];
    int dj = SPX_NONE;                                     // the Dantzig column of the CTA's first row with b < 0
    if (bneg != SPX_NONE) {
        unsigned long long d1[1] = {~0ull};
        for (int j = tid; j < m; j += nt) {
            const double v = own(bneg, j);
            if (v > 0.0) {
                const unsigned long long k = db_pos_key(v);
                if (k < d1[0]) { d1[0] = k; dj = j; }
            }
        }
        const unsigned long long my = d1[0];
        block_min_keys<1>(d1, red);
        unsigned long long j1[1] = {my == d1[0] && dj != SPX_NONE ? (unsigned long long)dj : ~0ull};
        block_min_keys<1>(j1, red);
        dj = j1[0] == ~0ull ? SPX_NONE : (int)j1[0];
    }
    if (tid == 0) part[0] = DbPartial{k2[0], s2[0], k2[1], dj, bneg == SPX_NONE ? SPX_NONE : r0 + bneg};
    cluster.sync();                                        // A

    int t = SPX_NONE;                                      // the target row (phase 1), the same in every CTA
    if (tid < 32) {
        DbPartial p{~0ull, ~0ull, ~0ull, SPX_NONE, SPX_NONE};
        if (lane < S) p = *cluster.map_shared_rank(&part[0], lane);
        const unsigned long long rk = warp_min_u64(p.rk), s = warp_min_u64(p.rk == rk ? p.sk : ~0ull);
        const unsigned long long bk = warp_min_u64(p.bk);
        t = warp_min_int(p.bneg);
        const int d = warp_min_int(p.bneg == t ? p.dj : SPX_NONE);   // from the owner of row t
        int st = SPX_PIVOT, rr = -1, cc = -1, next = -1;
        if (t != SPX_NONE) {
            if (d == SPX_NONE) st = SPX_INCORRECT; else next = d;   // phase 1: leave(c_D) in round 2
        } else if (cf == SPX_NONE) {
            st = SPX_OPTIMAL;
        } else if (rk == ~0ull) {
            st = SPX_NOCONV;                               // c_D is a ray
        } else if (rk != DB_ZERO_RATIO) {
            rr = (int)(s & 0x7fffffffu); cc = cf;
        } else {
            next = (int)(bk & 0xffffffffu);                // a degenerate step: Bland's column in round 2
        }
        if (lane == 0) { ctl[0] = st; ctl[1] = rr; ctl[2] = cc; ctl[3] = next; ctl[4] = t; }
    }
    __syncthreads();
    int st = ctl[0], next = ctl[3];
    r = ctl[1]; c = ctl[2];
    t = ctl[4];
    const int tf = t;                                      // SPX_NONE in phase 2: no row is the target

    // ---- rounds 2 and 3: the leaving row of column `next`; in round 2 of phase 1 also Bland's column of row t
    for (int round = 2; st == SPX_PIVOT && next >= 0; ++round) {
        DbPartial *mine_p = &part[(round - 1) & 1];     // round 2: part[1], round 3: part[0]
        const bool bland = tf != SPX_NONE && round == 2;
        unsigned long long k[2] = {~0ull, ~0ull};          // {ratio key, Bland key}
        unsigned long long s = ~0ull;
        for (int i = tid; i < rows; i += nt) db_leave_fold(k[0], s, r0 + i, own(i, next), own(i, m), tf, cl[i]);
        if (bland)
            for (int j = tid; j < cols; j += nt)
                if (row(tf, j0 + j) > 0.0) k[1] = min(k[1], db_label_key(rl[j], j0 + j));
        const unsigned long long my = k[0];
        block_min_keys<2>(k, red);
        unsigned long long s1[1] = {my == k[0] ? s : ~0ull};
        block_min_keys<1>(s1, red);
        if (tid == 0) *mine_p = DbPartial{k[0], s1[0], k[1], SPX_NONE, SPX_NONE};
        cluster.sync();                                    // A2 / A3
        if (tid < 32) {
            DbPartial p{~0ull, ~0ull, ~0ull, SPX_NONE, SPX_NONE};
            if (lane < S) p = *cluster.map_shared_rank(mine_p, lane);
            const unsigned long long rk = warp_min_u64(p.rk), sr = warp_min_u64(p.rk == rk ? p.sk : ~0ull);
            const unsigned long long bk = warp_min_u64(p.bk);
            int st2 = SPX_PIVOT, rr = -1, cc = -1, nx = -1;
            if (rk == ~0ull) {
                st2 = SPX_NOCONV;                          // phase 2 only: phase 1 always has its target
            } else if (bland && rk == DB_ZERO_RATIO) {
                nx = (int)(bk & 0xffffffffu);              // phase 1, a degenerate step: Bland's column in round 3
            } else {
                rr = (int)(sr & 0x7fffffffu); cc = next;
            }
            if (lane == 0) { ctl[0] = st2; ctl[1] = rr; ctl[2] = cc; ctl[3] = nx; }
        }
        __syncthreads();
        st = ctl[0]; next = ctl[3];
        r = ctl[1]; c = ctl[2];
    }
    return st;
}

// ---- host: the launch of a K7 or K8 kernel ----
// launch configuration of `clusters` LPs at S CTAs each with `smem` bytes of dynamic shared memory per CTA; attr must
// outlive cfg
inline cudaLaunchConfig_t cluster_launch_config(int64_t smem, int S, int64_t clusters, cudaLaunchAttribute *attr,
                                                cudaStream_t stream) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(clusters * S));
    cfg.blockDim = dim3(CLUSTER_THREADS);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = stream;
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)S;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cfg;
}

// one-time per-device set-up of Kernel's shared memory and cluster size limits
template <auto Kernel>
cudaError_t configure_cluster_kernel() {
    static bool configured_dev[64] = {};
    const int slot = spx_host::device_slot();
    if (configured_dev[slot]) return cudaSuccess;
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, Kernel);
    if (e != cudaSuccess) return e;
    if (fa.sharedSizeBytes > CLUSTER_STATIC) return cudaErrorInvalidValue;
    e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CLUSTER_DYN_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) return e;
    configured_dev[slot] = true;
    return cudaSuccess;
}

// Kernel(args...) on `clusters` LPs at S CTAs each (validated by the caller) with `smem` bytes per CTA; returns
// cudaErrorInvalidClusterSize when the device cannot co-schedule one such cluster
template <auto Kernel, typename... Args>
cudaError_t launch_cluster_kernel(int S, int64_t clusters, int64_t smem, cudaStream_t stream, Args... args) {
    if (clusters <= 0) return cudaSuccess;
    cudaError_t e = configure_cluster_kernel<Kernel>();
    if (e != cudaSuccess) return e;
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = cluster_launch_config(smem, S, clusters, attr, stream);
    int active = 0;
    e = cudaOccupancyMaxActiveClusters(&active, Kernel, &cfg);
    if (e != cudaSuccess) return e;
    if (active <= 0) return cudaErrorInvalidClusterSize;
    e = cudaLaunchKernelEx(&cfg, Kernel, args...);
    spx_host::count_launch();
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

} // namespace spx

// The arguments of the K7 and K8 kernels.  They live in the including file's anonymous namespace, with its kernels.
namespace {

struct ClusterArgs {
    double  *T;          // [B][cells] in/out
    int64_t  B;
    int      n, m, rule, max_pivots;
    int      S, R, Q;    // CTAs per LP, body rows per CTA, header labels per CTA
    double  *x;          // [B][m] or null
    double  *obj;        // [B] or null
    int32_t *status;     // [B]
    int32_t *npiv;       // [B]
    int32_t *rowlab;     // [B][m] or null
    int32_t *collab;     // [B][n] or null
    int32_t *trace;      // [B][max_pivots][2] or null
    double  *snap;       // [B][max_pivots+1][cells] or null
};

// B LPs of n x m at S CTAs each; a ragged launch passes n = m = max_pivots = 0 (its kernels read each LP's own)
inline ClusterArgs cluster_args(const spx::BatchIO &io, int64_t B, int n, int m, int S, int max_pivots) {
    return {io.T, B, n, m, io.rule, max_pivots, S, (n + S - 1) / S, (m + S - 1) / S,
            io.x, io.obj, io.status, io.npiv, io.rowlab, io.collab, io.trace, io.snap};
}

} // namespace
