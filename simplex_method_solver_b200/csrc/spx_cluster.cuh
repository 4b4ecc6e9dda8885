// spx_cluster.cuh — the pricing steps shared by the two one-cluster-per-LP solvers, K7 (spx_cluster.cu, table in
// shared memory) and K8 (spx_global.cu, table in global memory): the entering column of the replicated f row and
// the merge of the S per-CTA partials into one pivot decision that every CTA reaches on its own.
#pragma once
#include <cooperative_groups.h>

#include "spx_block.cuh"

namespace spx {

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

} // namespace spx
