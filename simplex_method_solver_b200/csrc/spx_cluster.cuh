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
