// spx_batched.cu — K4: whole-LP solver for batches of independent small LPs, no communication:
// the loop of get_solution(), /root/reference/src/simplex.py:179-199, with pick_element()
// (:70-141) and recalculate_matrix() (:143-177) inlined.
//
// The tableau of an LP lives in shared memory in the reference's own flat layout (n rows of m+1
// cells, then the f row with m cells) as two ping-pong copies, because the reference pivots out
// of place (:149) and every cell of the new table reads the OLD pivot row and column.
//   warp mode (<= 96 cells: cfg1 14 cells, cfg3 26 cells): one warp per LP, 8 LPs per CTA; every
//       decision is a warp ballot / redux, all 32 lanes take the same branch, __syncwarp only.
//   CTA mode (Klee-Minty n=20: 440 cells, 2^20-1 strictly sequential pivots): one CTA of 2..16 warps
//       per LP; warp 0 prices the pivot, every thread updates one cell (32 cells per warp), two block
//       barriers per pivot.
// The four cell kinds of the pivot differ only in the numerator, so one division by the pivot
// (pivot_div, reciprocal hoisted) serves them all without divergence.
#include "spx_launch.cuh"

namespace {

using namespace spx;

constexpr size_t SMEM_LIMIT = 227 * 1024;
constexpr int64_t CTA_MODE_MIN_CELLS = 96;    // above this one CTA (not one warp) solves an LP
constexpr int     CTA_CELLS_PER_WARP = 32;    // CTA mode: cells per warp (2..8 warps)
constexpr size_t  WARP_LUT_BYTES = CTA_MODE_MIN_CELLS * 4;   // ragged warp mode: per-warp lookup table (384 B)
constexpr size_t  K4_STATIC = 16;             // every K4 kernel: static shared memory (s_ctl), checked at launch
constexpr size_t  K4_DYN_LIMIT = SMEM_LIMIT - K4_STATIC;   // the dynamic and the static bytes of a CTA share SMEM_LIMIT

struct BatchedArgs {
    double  *T;          // [B][cells] in/out
    int64_t  B;
    int      n, m, rule, max_pivots;
    double  *x;          // [B][m] or null
    double  *obj;        // [B] or null
    int32_t *status;     // [B]
    int32_t *npiv;       // [B]
    int32_t *rowlab;     // [B][m] or null
    int32_t *collab;     // [B][n] or null
    int32_t *trace;      // [B][max_pivots][2] or null
    double  *snap;       // [B][max_pivots+1][cells] or null
};

// first index q in [0, len) with pred(q); warp-uniform result
template <class F>
__device__ __forceinline__ int warp_first_index(int len, int lane, F pred) {
    for (int base = 0; base < len; base += 32) {
        const int q = base + lane;
        const unsigned ball = __ballot_sync(0xffffffffu, q < len && pred(q));
        if (ball) return base + __ffs(ball) - 1;
    }
    return SPX_NONE;
}

// Cross-lane finish of the ratio scan.  Every lane holds the fold of its own rows; the decision of
// ratio_decide() over the union is taken with redux/ballot instead of a shuffle tree of structs.
__device__ __forceinline__ int warp_ratio_decide(const Ratio &q, bool my_elig_nan, int lane) {
    const unsigned full = 0xffffffffu;
    const int elig = __reduce_min_sync(full, q.elig_row);
    if (elig == SPX_NONE) return -1;                                       // first_try still True
    if (__ballot_sync(full, q.elig_row == elig && my_elig_nan)) return elig;   // NaN min_val is never replaced
    const bool has_neg = q.neg_row >= 0;
    if (__ballot_sync(full, has_neg)) {
        // largest negative ratio: max of the order-preserving 64-bit image, 32 bits at a time
        const unsigned long long key = has_neg ? orderable(q.neg_val) : 0ull;
        const unsigned hi = (unsigned)(key >> 32);
        const unsigned mhi = __reduce_max_sync(full, hi);
        const bool c1 = has_neg && hi == mhi;
        const unsigned lo = c1 ? (unsigned)key : 0u;
        const unsigned mlo = __reduce_max_sync(full, lo);
        const bool c2 = c1 && lo == mlo;
        return __reduce_max_sync(full, c2 ? q.neg_row : -1);               // ties -> highest row (:133, '<=')
    }
    const int zero = __reduce_min_sync(full, q.zero_row);
    return (zero != SPX_NONE) ? zero : -1;                                 // first zero ratio, else min_val > 0
}

// Devex entering column of the f row f[0..m) under the weights w (devex_key: the minimum of (key, j)); warp-uniform
__device__ __forceinline__ int warp_devex_entering(const double *f, const double *w, int m, int lane) {
    unsigned long long best = ~0ull;
    int bj = SPX_NONE;
    for (int j = lane; j < m; j += 32) {
        const double v = f[j];
        if (v < 0.0) {
            const unsigned long long k = devex_key(v, w[j]);
            if (k < best) { best = k; bj = j; }
        }
    }
    unsigned long long g = best;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, g, s);
        g = o < g ? o : g;
    }
    return __reduce_min_sync(0xffffffffu, best == g ? bj : SPX_NONE);
}

// The devex weights w[0..m) after pivot (r, c) of the table `cur`, by one warp in place.  u_j is the cell the update
// writes into the new pivot row; every lane reads w_c before any lane overwrites it.
__device__ __forceinline__ void warp_devex_update(const double *cur, double *w, int m, int r, int c, int lane) {
    const double *prow = cur + r * (m + 1);
    const PivotDiv d = pivot_div_prepare(prow[c]);
    const double wc = w[c];
    __syncwarp();
    for (int j = lane; j < m; j += 32)
        w[j] = devex_weight(w[j], pivot_div(j == c ? 1.0 : -prow[j], d), wc, j == c);
}

// K1 + K2 by ONE warp on the shared-memory table `cur`: returns SPX_PIVOT with (r, c) or the
// terminal status.  All 32 lanes take the same branches (ballots / redux only).  DEVEX: the entering column of
// phase 2 by the devex weights w (global memory) instead of `rule`.
template <bool DEVEX = false>
__device__ __forceinline__ int warp_pick(const double *cur, int n, int m, int rule, int lane, int &r, int &c,
                                         const double *w = nullptr) {
    const int w1 = m + 1, fo = n * w1;
    // ---- K1: phase-1 row (:72-76), its first positive cell (:81-85) ...
    const int r1 = warp_first_index(n, lane, [&](int i) { return cur[i * w1 + m] < 0.0; });
    if (r1 != SPX_NONE) {
        c = warp_first_index(m, lane, [&](int j) { return cur[r1 * w1 + j] > 0.0; });
        if (c == SPX_NONE) return SPX_INCORRECT;                                  // :88-89
        r = r1;                                                                   // :91
        return SPX_PIVOT;
    }
    // ---- ... or the entering column from the f row (:94-98)
    if constexpr (DEVEX) {
        c = warp_devex_entering(cur + fo, w, m, lane);
    } else if (rule == SPX_RULE_REFERENCE) {
        c = warp_first_index(m, lane, [&](int j) { return cur[fo + j] < 0.0; });
    } else {   // Dantzig: most negative, lowest index on ties
        unsigned long long best = ~0ull;
        for (int j = lane; j < m; j += 32) {
            const double v = cur[fo + j];
            if (v < 0.0) { const unsigned long long k = orderable(v); best = k < best ? k : best; }
        }
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            const unsigned long long o = __shfl_xor_sync(0xffffffffu, best, s);
            best = o < best ? o : best;
        }
        c = (best == ~0ull) ? SPX_NONE
            : warp_first_index(m, lane, [&](int j) {
                  const double v = cur[fo + j];
                  return v < 0.0 && orderable(v) == best; });
    }
    if (c == SPX_NONE) return SPX_OPTIMAL;                                        // :101-103
    // ---- K2: the ratio scan (:107-136): lane-local fold, then ballots / redux across lanes
    Ratio q = ratio_identity();
    bool my_elig_nan = false;                    // is the ratio of MY first eligible row NaN?
    for (int i = lane; i < n; i += 32) {
        const double a_ic = cur[i * w1 + c], b_i = cur[i * w1 + m];
        const bool first = (q.elig_row == SPX_NONE);
        const bool is_nan = ratio_accumulate(q, i, a_ic, b_i);
        if (first && q.elig_row != SPX_NONE) my_elig_nan = is_nan;
    }
    r = warp_ratio_decide(q, my_elig_nan, lane);
    return (r < 0) ? SPX_NOCONV : SPX_PIVOT;                                      // :138-139
}

__device__ __forceinline__ unsigned long long warp_min_key(unsigned long long v) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, v, s);
        v = o < v ? o : v;
    }
    return v;
}

// SPX_RULE_DANTZIG_BLAND's leaving row of column c by one warp (t: the target row, SPX_NONE in phase 2; cl: the row
// labels); -1 when no row is a candidate, rk = its ratio key; warp-uniform
__device__ __forceinline__ int warp_db_leave(const double *cur, int n, int m, int c, int t, const int32_t *cl, int lane,
                                             unsigned long long &rk) {
    const int w1 = m + 1;
    unsigned long long k = ~0ull, s = ~0ull;
    for (int i = lane; i < n; i += 32) db_leave_fold(k, s, i, cur[i * w1 + c], cur[i * w1 + m], t, cl[i]);
    rk = warp_min_key(k);
    s = warp_min_key(k == rk ? s : ~0ull);
    return rk == ~0ull ? -1 : (int)(s & 0x7fffffffu);
}

// K1 + K2 under SPX_RULE_DANTZIG_BLAND by ONE warp on `cur` with its header labels rl and row labels cl: returns
// SPX_PIVOT with (r, c) or the terminal status; warp-uniform
__device__ __forceinline__ int warp_pick_db(const double *cur, int n, int m, const int32_t *rl, const int32_t *cl,
                                            int lane, int &r, int &c) {
    const int w1 = m + 1;
    const int t = warp_first_index(n, lane, [&](int i) { return cur[i * w1 + m] < 0.0; });
    const bool ph1 = t != SPX_NONE;
    const double *e = cur + (ph1 ? t : n) * w1;           // phase 1: row t; phase 2: the f row
    unsigned long long dk = ~0ull, bk = ~0ull;            // Dantzig's key and Bland's key of this lane's candidates
    int dj = SPX_NONE;
    for (int j = lane; j < m; j += 32) {
        const double v = e[j];
        if (ph1 ? v > 0.0 : v < 0.0) {
            const unsigned long long k = ph1 ? db_pos_key(v) : orderable(v);
            if (k < dk) { dk = k; dj = j; }
            const unsigned long long b = db_label_key(rl[j], j);
            bk = b < bk ? b : bk;
        }
    }
    const unsigned long long g = warp_min_key(dk);
    if (g == ~0ull) return ph1 ? SPX_INCORRECT : SPX_OPTIMAL;
    c = __reduce_min_sync(0xffffffffu, dk == g ? dj : SPX_NONE);
    unsigned long long rk;
    r = warp_db_leave(cur, n, m, c, t, cl, lane, rk);
    if (r >= 0 && rk == DB_ZERO_RATIO) {                   // a degenerate step: Bland's column and its leaving row
        c = (int)(warp_min_key(bk) & 0xffffffffu);
        r = warp_db_leave(cur, n, m, c, t, cl, lane, rk);
    }
    return r < 0 ? SPX_NOCONV : SPX_PIVOT;
}

// K1 + K2 of batched_solve / ragged_body: DB selects SPX_RULE_DANTZIG_BLAND, else warp_pick<DEVEX>
template <bool DEVEX, bool DB>
__device__ __forceinline__ int warp_pick_any(const double *cur, int n, int m, int rule, int lane, int &r, int &c,
                                             const double *w, const int32_t *rl, const int32_t *cl) {
    if constexpr (DB) return warp_pick_db(cur, n, m, rl, cl, lane, r, c);
    else return warp_pick<DEVEX>(cur, n, m, rule, lane, r, c, w);
}

// CTA == false: one warp per LP, warps_per_cta LPs per CTA, __syncwarp between the phases
//               (cfg1: 14 cells, cfg3: 26 cells — one cell per lane).
// CTA == true : one CTA per LP for tables of hundreds of cells (Klee-Minty n=20: 440 cells, 2^20-1
//               strictly sequential pivots): warp 0 prices the pivot, every warp updates its share
//               of the cells, two block barriers per pivot.
// is `lab` the label of a variable x_(lab+1)?  A resume also rejects negative labels (it never indexes with one)
template <bool WARM>
__device__ __forceinline__ bool x_label(int lab, int m) {
    if constexpr (WARM) return lab >= 0 && lab < m;
    else return lab < m;
}

// CTA == false / true as above.
// WARM == false: a solve from the loaded table, labels 'x1'..'xm' / 'y1'..'yn', f0 and f1 from its f row.
// WARM == true:  a resume (spx_warm_solve_batched): labels read from a.rowlab / a.collab, f0 and f1 for obj from
//                `function` [B][m], and no label outside [0, m) indexes xs.

// DEVEX: the devex rule (SPX_RULE_DEVEX) with the weights in the LP's x slice, a.x[lp][0..m): set to 1 here, updated
// by the warp that prices, after each pick, and overwritten by x in the epilogue.
template <bool CTA, bool WARM, bool DEVEX = false, bool DB = false>
__device__ __forceinline__ void batched_solve(const BatchedArgs &a, const double *function, int warps_per_cta,
                                              int warp_doubles) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_ctl[4];                               // CTA mode: {status, r, c} of warp 0's pick
    const int n = a.n, m = a.m, w1 = m + 1;
    const int cells = n * w1 + m;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    // CTA-shared lookup: cell -> (row, col), built once (shape is uniform over the batch)
    uint16_t *cell_i = reinterpret_cast<uint16_t *>(smem_raw);
    uint16_t *cell_j = cell_i + cells;
    for (int k = threadIdx.x; k < cells; k += blockDim.x) {
        const int i = k / w1;
        cell_i[k] = (uint16_t)i;
        cell_j[k] = (uint16_t)(k - i * w1);
    }
    __syncthreads();

    const int64_t lp = CTA ? (int64_t)blockIdx.x : (int64_t)blockIdx.x * warps_per_cta + warp;
    if (!CTA && (warp >= warps_per_cta || lp >= a.B)) return;
    // a resume: the current costs for obj, read before anything else (read later, around the label loads or in the
    // epilogue, they cost warp mode, at the register cap of its launch bounds, more spills than the solve has)
    const double c0 = (WARM && function && m >= 2) ? function[lp * m] : 0.0;
    const double c1 = (WARM && function && m >= 2) ? function[lp * m + 1] : 0.0;
    const int tl = CTA ? (int)threadIdx.x : lane;          // thread index within the LP's group
    const int nl = CTA ? (int)blockDim.x : 32;             // threads of the group
    auto group_sync = [&]() { if (CTA) __syncthreads(); else __syncwarp(); };

    const size_t lut_bytes = ((size_t)cells * 4 + 15) / 16 * 16;
    double *base = reinterpret_cast<double *>(smem_raw + lut_bytes) + (size_t)(CTA ? 0 : warp) * warp_doubles;
    double *cur = base;
    double *nxt = base + cells;
    double *xs  = base + 2 * cells;                       // [m]
    int32_t *rl = reinterpret_cast<int32_t *>(xs + m);    // [m] header labels
    int32_t *cl = rl + m;                                 // [n] row labels

    double *Tg = a.T + lp * (int64_t)cells;
    for (int k = tl; k < cells; k += nl) cur[k] = Tg[k];
    double *w = DEVEX ? a.x + lp * m : nullptr;
    if constexpr (DEVEX) for (int j = tl; j < m; j += nl) w[j] = 1.0;
    if constexpr (WARM) {
        for (int j = tl; j < m; j += nl) rl[j] = a.rowlab[lp * m + j];
        for (int i = tl; i < n; i += nl) cl[i] = a.collab[lp * n + i];
    } else {
        for (int j = tl; j < m; j += nl) rl[j] = j;       // 'x1'..'xm'  :30
        for (int i = tl; i < n; i += nl) cl[i] = m + i;   // 'y1'..'yn'  :31
    }
    group_sync();
    const int fo = n * w1;                                // offset of the f row
    const double f0 = (m >= 1) ? cur[fo] : 0.0;           // self.function is never mutated (:29,:49)
    const double f1 = (m >= 2) ? cur[fo + 1] : 0.0;

    int npiv = 0, status;
    double *snap = a.snap ? a.snap + lp * (int64_t)(a.max_pivots + 1) * cells : nullptr;
    int32_t *trace = a.trace ? a.trace + lp * (int64_t)a.max_pivots * 2 : nullptr;

    for (;;) {
        if (snap) {
            double *sg = snap + (int64_t)npiv * cells;
            for (int k = tl; k < cells; k += nl) sg[k] = cur[k];
        }
        int r = -1, c = -1;
        if (!CTA) {
            status = warp_pick_any<DEVEX, DB>(cur, n, m, a.rule, lane, r, c, w, rl, cl);
            if (DEVEX && status == SPX_PIVOT) warp_devex_update(cur, w, m, r, c, lane);
        } else {
            if (warp == 0) {
                const int st = warp_pick_any<DEVEX, DB>(cur, n, m, a.rule, lane, r, c, w, rl, cl);
                if (DEVEX && st == SPX_PIVOT) warp_devex_update(cur, w, m, r, c, lane);
                if (lane == 0) { s_ctl[0] = st; s_ctl[1] = r; s_ctl[2] = c; }
            }
            __syncthreads();
            status = s_ctl[0]; r = s_ctl[1]; c = s_ctl[2];
        }
        if (status != SPX_PIVOT) break;
        if (npiv >= a.max_pivots) { status = SPX_CAP; break; }
        if (trace && tl == 0) { trace[2 * npiv] = r; trace[2 * npiv + 1] = c; }

        // ---- K3: out-of-place pivot (:149-177), all reads from `cur`; the four cell kinds
        // (:156 pivot row, :160 pivot column, :163 pivot cell, :173-175 the rest) differ only in
        // the numerator, so one division by the pivot serves them all without divergence
        const double p = cur[r * w1 + c];
        const PivotDiv d = pivot_div_prepare(p);
        const double *prow = cur + r * w1;
        for (int k = tl; k < cells; k += nl) {
            const int i = cell_i[k], j = cell_j[k];
            const double t = cur[k];
            const double ci = cur[i * w1 + c];
            const bool pr = (i == r), pc = (j == c);
            double num = __dsub_rn(__dmul_rn(t, p), __dmul_rn(prow[j], ci));
            num = pc ? ci : num;
            num = pr ? -t : num;
            num = (pr && pc) ? 1.0 : num;
            nxt[k] = pivot_div(num, d);
        }
        if (tl == 0) { const int32_t t = rl[c]; rl[c] = cl[r]; cl[r] = t; }      // :152
        group_sync();                                      // (CTA: also orders s_ctl against the next pick)
        double *sw = cur; cur = nxt; nxt = sw;
        ++npiv;
    }

    // ---- epilogue: final table, labels, find_optimum()/f() (:48-68)
    for (int k = tl; k < cells; k += nl) Tg[k] = cur[k];
    for (int j = tl; j < m; j += nl) xs[j] = 0.0;
    group_sync();
    for (int i = tl; i < n; i += nl) {
        const int lab = cl[i];
        if (x_label<WARM>(lab, m)) xs[lab] = cur[i * w1 + m];
    }
    group_sync();
    if (a.x) for (int j = tl; j < m; j += nl) a.x[lp * m + j] = xs[j];
    if (a.rowlab) for (int j = tl; j < m; j += nl) a.rowlab[lp * m + j] = rl[j];
    if (a.collab) for (int i = tl; i < n; i += nl) a.collab[lp * n + i] = cl[i];
    if (tl == 0) {
        a.status[lp] = status;
        a.npiv[lp] = npiv;
        if (a.obj) a.obj[lp] = (m >= 2) ? __dadd_rn(__dmul_rn(WARM ? c0 : f0, xs[0]), __dmul_rn(WARM ? c1 : f1, xs[1])) : 0.0;
    }
}

template <bool CTA>
__global__ void __launch_bounds__(CTA ? 512 : 256, CTA ? 1 : 6)
batched_kernel(BatchedArgs a, int warps_per_cta, int warp_doubles) {
    batched_solve<CTA, false>(a, nullptr, warps_per_cta, warp_doubles);
}

// the resume of batched_kernel (spx_warm_solve_batched); function [B][m], the LPs' current costs, or null without obj
template <bool CTA>
__global__ void __launch_bounds__(CTA ? 512 : 256, CTA ? 1 : 6)
batched_warm_kernel(BatchedArgs a, const double *function, int warps_per_cta, int warp_doubles) {
    batched_solve<CTA, true>(a, function, warps_per_cta, warp_doubles);
}

// batched_kernel (WARM == false, function null) and batched_warm_kernel (WARM == true) under the devex rule
template <bool CTA, bool WARM>
__global__ void __launch_bounds__(CTA ? 512 : 256, CTA ? 1 : 6)
batched_devex_kernel(BatchedArgs a, const double *function, int warps_per_cta, int warp_doubles) {
    batched_solve<CTA, WARM, true>(a, function, warps_per_cta, warp_doubles);
}

// batched_kernel (WARM == false, function null) and batched_warm_kernel (WARM == true) under SPX_RULE_DANTZIG_BLAND
template <bool CTA, bool WARM>
__global__ void __launch_bounds__(CTA ? 512 : 256, CTA ? 1 : 6)
batched_db_kernel(BatchedArgs a, const double *function, int warps_per_cta, int warp_doubles) {
    batched_solve<CTA, WARM, false, true>(a, function, warps_per_cta, warp_doubles);
}

// One LP of a ragged batch, start to finish: batched_kernel's loop with the shape and the offsets taken from the LP's
// descriptor `d`, by its group of nl threads (tl = index in the group): one warp (CTA == false) or the first nl
// threads of the CTA (CTA == true).  base: its two tables, x, labels in shared memory.  In warp mode the warps of one
// CTA have different shapes, so each warp has its own cell -> (row, col) lookup table (cell_i, cell_j) instead of a
// CTA-wide one; in CTA mode the group synchronises with a named barrier of its own nl threads.
// (batched_kernel keeps its own copy of the loop: it runs at the 40-register cap of its launch bounds in warp mode,
// and any restructuring of its code moves its spills.)  WARM: the resume, as batched_solve's; gd: LP lp's descriptor
// in global memory (d is its copy).
template <bool CTA, bool WARM, bool DEVEX, bool DB = false>
__device__ __forceinline__ void ragged_body(const BatchedArgs &a, const RaggedLp &d, int64_t lp, const uint16_t *cell_i,
                                             const uint16_t *cell_j, double *base, int *s_ctl, int tl, int nl,
                                             const double *function, const RaggedLp *gd) {
    const int n = d.n, m = d.m, w1 = m + 1;
    const int cells = n * w1 + m;
    const int max_pivots = d.max_pivots;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    auto group_sync = [&]() {
        if (!CTA) __syncwarp();
        else asm volatile("bar.sync 1, %0;" :: "r"(nl) : "memory");
    };

    double *cur = base;
    double *nxt = base + cells;
    double *xs  = base + 2 * cells;                       // [m]
    int32_t *rl = reinterpret_cast<int32_t *>(xs + m);    // [m] header labels
    int32_t *cl = rl + m;                                 // [n] row labels

    double *Tg = a.T + d.t;
    for (int k = tl; k < cells; k += nl) cur[k] = Tg[k];
    double *w = DEVEX ? a.x + d.xm : nullptr;            // batched_solve's devex weights, in the LP's x slice
    if constexpr (DEVEX) for (int j = tl; j < m; j += nl) w[j] = 1.0;
    double c0 = 0.0, c1 = 0.0;                            // a resume: the current costs for obj
    if constexpr (WARM) {
        // The offsets come from the descriptor in global memory (gd, read once each), not from d: warp mode runs at
        // the register cap of its launch bounds and keeps d's offsets in local memory, so reading them there would
        // cost more spill loads than the solve has.
        const int64_t xm = *(volatile const int64_t *)&gd->xm, xn = *(volatile const int64_t *)&gd->xn;
        for (int j = tl; j < m; j += nl) rl[j] = a.rowlab[xm + j];
        if (function && m >= 2) { c0 = function[xm]; c1 = function[xm + 1]; }
        for (int i = tl; i < n; i += nl) cl[i] = a.collab[xn + i];
    } else {
        for (int j = tl; j < m; j += nl) rl[j] = j;       // 'x1'..'xm'  :30
        for (int i = tl; i < n; i += nl) cl[i] = m + i;   // 'y1'..'yn'  :31
    }
    group_sync();
    const int fo = n * w1;                                // offset of the f row
    const double f0 = (m >= 1) ? cur[fo] : 0.0;           // self.function is never mutated (:29,:49)
    const double f1 = (m >= 2) ? cur[fo + 1] : 0.0;

    int npiv = 0, status;
    double *snap = a.snap ? a.snap + d.sn : nullptr;
    int32_t *trace = a.trace ? a.trace + 2 * d.tr : nullptr;

    for (;;) {
        if (snap) {
            double *sg = snap + (int64_t)npiv * cells;
            for (int k = tl; k < cells; k += nl) sg[k] = cur[k];
        }
        int r = -1, c = -1;
        if (!CTA) {
            status = warp_pick_any<DEVEX, DB>(cur, n, m, a.rule, lane, r, c, w, rl, cl);
            if (DEVEX && status == SPX_PIVOT) warp_devex_update(cur, w, m, r, c, lane);
        } else {
            if (warp == 0) {
                const int st = warp_pick_any<DEVEX, DB>(cur, n, m, a.rule, lane, r, c, w, rl, cl);
                if (DEVEX && st == SPX_PIVOT) warp_devex_update(cur, w, m, r, c, lane);
                if (lane == 0) { s_ctl[0] = st; s_ctl[1] = r; s_ctl[2] = c; }
            }
            group_sync();
            status = s_ctl[0]; r = s_ctl[1]; c = s_ctl[2];
        }
        if (status != SPX_PIVOT) break;
        if (npiv >= max_pivots) { status = SPX_CAP; break; }
        if (trace && tl == 0) { trace[2 * npiv] = r; trace[2 * npiv + 1] = c; }

        // ---- K3: out-of-place pivot (:149-177), all reads from `cur`; the four cell kinds
        // (:156 pivot row, :160 pivot column, :163 pivot cell, :173-175 the rest) differ only in
        // the numerator, so one division by the pivot serves them all without divergence
        const double p = cur[r * w1 + c];
        const PivotDiv pd = pivot_div_prepare(p);
        const double *prow = cur + r * w1;
        for (int k = tl; k < cells; k += nl) {
            const int i = cell_i[k], j = cell_j[k];
            const double t = cur[k];
            const double ci = cur[i * w1 + c];
            const bool pr = (i == r), pc = (j == c);
            double num = __dsub_rn(__dmul_rn(t, p), __dmul_rn(prow[j], ci));
            num = pc ? ci : num;
            num = pr ? -t : num;
            num = (pr && pc) ? 1.0 : num;
            nxt[k] = pivot_div(num, pd);
        }
        if (tl == 0) { const int32_t t = rl[c]; rl[c] = cl[r]; cl[r] = t; }      // :152
        group_sync();                                      // (CTA: also orders s_ctl against the next pick)
        double *sw = cur; cur = nxt; nxt = sw;
        ++npiv;
    }

    // ---- epilogue: final table, labels, find_optimum()/f() (:48-68)
    for (int k = tl; k < cells; k += nl) Tg[k] = cur[k];
    for (int j = tl; j < m; j += nl) xs[j] = 0.0;
    group_sync();
    for (int i = tl; i < n; i += nl) {
        const int lab = cl[i];
        if (x_label<WARM>(lab, m)) xs[lab] = cur[i * w1 + m];
    }
    group_sync();
    if (a.x) for (int j = tl; j < m; j += nl) a.x[d.xm + j] = xs[j];
    if (a.rowlab) for (int j = tl; j < m; j += nl) a.rowlab[d.xm + j] = rl[j];
    if (a.collab) for (int i = tl; i < n; i += nl) a.collab[d.xn + i] = cl[i];
    if (tl == 0) {
        a.status[lp] = status;
        a.npiv[lp] = npiv;
        if (a.obj) a.obj[lp] = (m >= 2) ? __dadd_rn(__dmul_rn(WARM ? c0 : f0, xs[0]), __dmul_rn(WARM ? c1 : f1, xs[1])) : 0.0;
    }
}

// The ragged batch: LP order[slot] of each slot, shape and offsets from lps[].  Warp mode: slot = warp of the grid,
// warp slots of warp_doubles doubles, each a 384-byte lookup table and then the LP's tables, x and labels; same launch
// bounds as batched_kernel<false>.  CTA mode: slot = CTA; the CTA is launched at the warp count of
// the largest LP of the launch, builds the lookup table of its own LP, and only the warps its LP needs stay (the
// warp count the uniform entry gives that shape: 32 cells per warp, 2..16 warps).
template <bool CTA, bool WARM, bool DEVEX = false, bool DB = false>
__device__ __forceinline__ void ragged_batched(const BatchedArgs &a, const RaggedLp *__restrict__ lps,
                                               const int32_t *__restrict__ order, int warps_per_cta, int warp_doubles,
                                               const double *function) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_ctl[4];
    const int warp = threadIdx.x >> 5;
    const int64_t slot = CTA ? (int64_t)blockIdx.x : (int64_t)blockIdx.x * warps_per_cta + warp;
    if (!CTA) {
        if (warp >= warps_per_cta || slot >= a.B) return;
        const int64_t lp = order[slot];
        const RaggedLp d = lps[lp];
        const int lane = threadIdx.x & 31, w1 = d.m + 1;
        // the warp's slot: its own lookup table (<= 96 cells), then its tables, x and labels
        unsigned char *slot_raw = smem_raw + (size_t)warp * warp_doubles * sizeof(double);
        uint16_t *cell_i = reinterpret_cast<uint16_t *>(slot_raw);
        uint16_t *cell_j = cell_i + CTA_MODE_MIN_CELLS;
        for (int k = lane; k < d.cells; k += 32) {
            const int i = k / w1;
            cell_i[k] = (uint16_t)i;
            cell_j[k] = (uint16_t)(k - i * w1);
        }
        __syncwarp();
        double *base = reinterpret_cast<double *>(slot_raw + WARP_LUT_BYTES);
        ragged_body<false, WARM, DEVEX, DB>(a, d, lp, cell_i, cell_j, base, s_ctl, lane, 32, function, lps + lp);
        return;
    }
    const int64_t lp = order[slot];
    const RaggedLp d = lps[lp];
    const int w1 = d.m + 1, cells = d.cells;
    uint16_t *cell_i = reinterpret_cast<uint16_t *>(smem_raw);
    uint16_t *cell_j = cell_i + cells;
    for (int k = threadIdx.x; k < cells; k += blockDim.x) {
        const int i = k / w1;
        cell_i[k] = (uint16_t)i;
        cell_j[k] = (uint16_t)(k - i * w1);
    }
    __syncthreads();
    int warps = (cells + CTA_CELLS_PER_WARP - 1) / CTA_CELLS_PER_WARP;
    warps = warps < 2 ? 2 : (warps > 16 ? 16 : warps);
    const int nl = warps * 32 < (int)blockDim.x ? warps * 32 : (int)blockDim.x;
    if ((int)threadIdx.x >= nl) return;
    const size_t lut_bytes = ((size_t)cells * 4 + 15) / 16 * 16;
    double *base = reinterpret_cast<double *>(smem_raw + lut_bytes);
    ragged_body<true, WARM, DEVEX, DB>(a, d, lp, cell_i, cell_j, base, s_ctl, (int)threadIdx.x, nl, function, lps + lp);
}

template <bool CTA>
__global__ void __launch_bounds__(CTA ? 512 : 256, CTA ? 1 : 6)
ragged_batched_kernel(BatchedArgs a, const RaggedLp *__restrict__ lps, const int32_t *__restrict__ order,
                      int warps_per_cta, int warp_doubles) {
    ragged_batched<CTA, false>(a, lps, order, warps_per_cta, warp_doubles, nullptr);
}

// the resume of ragged_batched_kernel (spx_warm_solve_ragged); function packed as x, or null without obj
template <bool CTA>
__global__ void __launch_bounds__(CTA ? 512 : 256, CTA ? 1 : 6)
ragged_batched_warm_kernel(BatchedArgs a, const RaggedLp *__restrict__ lps, const int32_t *__restrict__ order,
                           int warps_per_cta, int warp_doubles, const double *function) {
    ragged_batched<CTA, true>(a, lps, order, warps_per_cta, warp_doubles, function);
}

// ragged_batched_kernel (WARM == false, function null) and ragged_batched_warm_kernel (WARM == true) under the devex rule
template <bool CTA, bool WARM>
__global__ void __launch_bounds__(CTA ? 512 : 256, CTA ? 1 : 6)
ragged_batched_devex_kernel(BatchedArgs a, const RaggedLp *__restrict__ lps, const int32_t *__restrict__ order,
                            int warps_per_cta, int warp_doubles, const double *function) {
    ragged_batched<CTA, WARM, true>(a, lps, order, warps_per_cta, warp_doubles, function);
}

// ragged_batched_kernel (WARM == false, function null) and ragged_batched_warm_kernel (WARM == true) under
// SPX_RULE_DANTZIG_BLAND
template <bool CTA, bool WARM>
__global__ void __launch_bounds__(CTA ? 512 : 256, CTA ? 1 : 6)
ragged_batched_db_kernel(BatchedArgs a, const RaggedLp *__restrict__ lps, const int32_t *__restrict__ order,
                         int warps_per_cta, int warp_doubles, const double *function) {
    ragged_batched<CTA, WARM, false, true>(a, lps, order, warps_per_cta, warp_doubles, function);
}

size_t warp_bytes(int n, int m) {
    const size_t cells = (size_t)n * (m + 1) + m;
    size_t b = (2 * cells + m) * sizeof(double) + (size_t)(n + m) * sizeof(int32_t);
    return (b + 15) / 16 * 16;
}
size_t lut_bytes(int n, int m) {
    const size_t cells = (size_t)n * (m + 1) + m;
    return (cells * 4 + 15) / 16 * 16;
}

// Kernel<<<grid, threads, smem, stream>>>(args...), counted.  Above 48 KB of dynamic shared memory the kernel's limit
// is first set to K4_DYN_LIMIT, once per device, after checking that its static bytes are the K4_STATIC the capacity
// rule reserves.  A failure of that set-up is returned once: the runtime's last error is cleared, so that the next
// launch's cudaGetLastError() does not report it again.
template <auto Kernel, typename... Args>
cudaError_t launch_k4(int64_t grid, int threads, size_t smem, cudaStream_t stream, Args... args) {
    static bool configured_dev[64] = {};
    bool &configured = configured_dev[spx_host::device_slot()];
    if (smem > 48 * 1024 && !configured) {
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, Kernel);
        if (e == cudaSuccess && fa.sharedSizeBytes > K4_STATIC) return cudaErrorInvalidValue;
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K4_DYN_LIMIT);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return e;
        }
        configured = true;
    }
    Kernel<<<(unsigned)grid, threads, smem, stream>>>(args...);
    spx_host::count_launch();
    return cudaGetLastError();
}

} // namespace

namespace spx_launch {

int64_t batched_max_cells() { return 10000; }

// K4's capacity, one rule for the uniform and the ragged entries: at most batched_max_cells() cells, and in CTA mode
// (above 96 cells) the lookup table and the LP's tables within K4_DYN_LIMIT; warp mode always fits
bool batched_fits(int n, int m) {
    if (n < 1 || m < 1 || n > 65535 || m > 65534) return false;
    const int64_t cells = (int64_t)n * (m + 1) + m;
    if (cells > batched_max_cells()) return false;
    return cells <= CTA_MODE_MIN_CELLS || lut_bytes(n, m) + warp_bytes(n, m) <= K4_DYN_LIMIT;
}

// returns cudaErrorInvalidValue when one LP does not fit shared memory; io.warm: the resume (batched_warm_kernel)
cudaError_t solve_batched(int64_t B, int n, int m, int max_pivots, const BatchIO &io, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    if (!batched_fits(n, m)) return cudaErrorInvalidValue;
    const size_t wb = warp_bytes(n, m), lb = lut_bytes(n, m);
    const int wd = (int)(wb / sizeof(double));
    const int64_t cells = (int64_t)n * (m + 1) + m;
    const BatchedArgs a{io.T, B, n, m, io.rule, max_pivots, io.x, io.obj, io.status, io.npiv, io.rowlab, io.collab,
                        io.trace, io.snap};
    if (cells > CTA_MODE_MIN_CELLS) {
        // one CTA per LP: one cell per thread where possible (measured on Klee-Minty n=20: 32 cells per warp
        // 891 k pivots/s, 64: 730 k, 128: 623 k), 2..16 warps
        int warps = (int)((cells + CTA_CELLS_PER_WARP - 1) / CTA_CELLS_PER_WARP);
        warps = warps < 2 ? 2 : (warps > 16 ? 16 : warps);
        if (io.rule == SPX_RULE_DEVEX)
            return io.warm ? launch_k4<batched_devex_kernel<true, true>>(B, warps * 32, lb + wb, stream, a, io.function, 1, wd)
                           : launch_k4<batched_devex_kernel<true, false>>(B, warps * 32, lb + wb, stream, a, nullptr, 1, wd);
        if (io.rule == SPX_RULE_DANTZIG_BLAND)
            return io.warm ? launch_k4<batched_db_kernel<true, true>>(B, warps * 32, lb + wb, stream, a, io.function, 1, wd)
                           : launch_k4<batched_db_kernel<true, false>>(B, warps * 32, lb + wb, stream, a, nullptr, 1, wd);
        if (io.warm) return launch_k4<batched_warm_kernel<true>>(B, warps * 32, lb + wb, stream, a, io.function, 1, wd);
        return launch_k4<batched_kernel<true>>(B, warps * 32, lb + wb, stream, a, 1, wd);
    }
    // warps per CTA: as many as fit ~48 KB (several CTAs per SM), at most 8, at least 1
    int wpc = (int)((48 * 1024 - lb) / wb);
    if (lb >= 48 * 1024) wpc = 0;
    wpc = wpc > 8 ? 8 : wpc;
    if (wpc < 1) wpc = 1;
    if ((int64_t)wpc > B) wpc = (int)B;
    const size_t smem = lb + (size_t)wpc * wb;
    const int64_t ctas = (B + wpc - 1) / wpc;
    if (io.rule == SPX_RULE_DEVEX)
        return io.warm ? launch_k4<batched_devex_kernel<false, true>>(ctas, wpc * 32, smem, stream, a, io.function, wpc, wd)
                       : launch_k4<batched_devex_kernel<false, false>>(ctas, wpc * 32, smem, stream, a, nullptr, wpc, wd);
    if (io.rule == SPX_RULE_DANTZIG_BLAND)
        return io.warm ? launch_k4<batched_db_kernel<false, true>>(ctas, wpc * 32, smem, stream, a, io.function, wpc, wd)
                       : launch_k4<batched_db_kernel<false, false>>(ctas, wpc * 32, smem, stream, a, nullptr, wpc, wd);
    if (io.warm) return launch_k4<batched_warm_kernel<false>>(ctas, wpc * 32, smem, stream, a, io.function, wpc, wd);
    return launch_k4<batched_kernel<false>>(ctas, wpc * 32, smem, stream, a, wpc, wd);
}

// ---- ragged batches: the plan's numbers for K4 ----
// shared memory of one LP: CTA mode lookup table + tables, or warp mode slot (no table); -1 when K4 cannot take it
// (batched_fits, the uniform entry's rule)
int64_t ragged_batched_bytes(int n, int m, int *kernel) {
    if (!batched_fits(n, m)) return -1;
    const int64_t cells = (int64_t)n * (m + 1) + m;
    *kernel = cells > CTA_MODE_MIN_CELLS ? RAGGED_CTA : RAGGED_WARP;
    return cells > CTA_MODE_MIN_CELLS ? (int64_t)(lut_bytes(n, m) + warp_bytes(n, m))
                                      : (int64_t)(WARP_LUT_BYTES + warp_bytes(n, m));
}
// CTA mode: the uniform entry's warp count for this many cells (32 cells per warp, 2..16 warps)
int ragged_cta_threads(int64_t cells) {
    int warps = (int)((cells + CTA_CELLS_PER_WARP - 1) / CTA_CELLS_PER_WARP);
    return 32 * (warps < 2 ? 2 : (warps > 16 ? 16 : warps));
}
// warp mode: LPs per CTA for warp slots of `slot` bytes (the lookup table included), as the uniform entry (at most 8, ~48 KB per CTA)
int ragged_warps_per_cta(int64_t slot, int64_t count) {
    int64_t wpc = (48 * 1024) / slot;
    wpc = wpc > 8 ? 8 : (wpc < 1 ? 1 : wpc);
    return (int)(wpc > count ? count : wpc);
}

cudaError_t solve_ragged_batched(const PlanView &v, const RaggedLaunch &l, const BatchIO &io, cudaStream_t stream) {
    if (l.count <= 0) return cudaSuccess;
    const BatchedArgs a{io.T, l.count, 0, 0, io.rule, 0, io.x, io.obj, io.status, io.npiv, io.rowlab, io.collab,
                        io.trace, io.snap};
    const int64_t ctas = (l.count + l.per_cta - 1) / l.per_cta;
    const size_t smem = (size_t)l.smem;
    const int32_t *order = v.d_order + l.first;
    const double *fn = io.warm ? io.function : nullptr;
    if (io.rule == SPX_RULE_DEVEX) {
        if (l.kernel == RAGGED_CTA)
            return io.warm ? launch_k4<ragged_batched_devex_kernel<true, true>>(ctas, l.threads, smem, stream, a, v.d_lps,
                                                                               order, 1, 0, fn)
                           : launch_k4<ragged_batched_devex_kernel<true, false>>(ctas, l.threads, smem, stream, a, v.d_lps,
                                                                                order, 1, 0, fn);
        return io.warm ? launch_k4<ragged_batched_devex_kernel<false, true>>(ctas, l.threads, smem, stream, a, v.d_lps,
                                                                            order, l.per_cta, (int)l.slot_doubles, fn)
                       : launch_k4<ragged_batched_devex_kernel<false, false>>(ctas, l.threads, smem, stream, a, v.d_lps,
                                                                             order, l.per_cta, (int)l.slot_doubles, fn);
    }
    if (io.rule == SPX_RULE_DANTZIG_BLAND) {
        if (l.kernel == RAGGED_CTA)
            return io.warm ? launch_k4<ragged_batched_db_kernel<true, true>>(ctas, l.threads, smem, stream, a, v.d_lps,
                                                                            order, 1, 0, fn)
                           : launch_k4<ragged_batched_db_kernel<true, false>>(ctas, l.threads, smem, stream, a, v.d_lps,
                                                                             order, 1, 0, fn);
        return io.warm ? launch_k4<ragged_batched_db_kernel<false, true>>(ctas, l.threads, smem, stream, a, v.d_lps,
                                                                         order, l.per_cta, (int)l.slot_doubles, fn)
                       : launch_k4<ragged_batched_db_kernel<false, false>>(ctas, l.threads, smem, stream, a, v.d_lps,
                                                                          order, l.per_cta, (int)l.slot_doubles, fn);
    }
    if (l.kernel == RAGGED_CTA)
        return io.warm ? launch_k4<ragged_batched_warm_kernel<true>>(ctas, l.threads, smem, stream, a, v.d_lps, order,
                                                                     1, 0, io.function)
                       : launch_k4<ragged_batched_kernel<true>>(ctas, l.threads, smem, stream, a, v.d_lps, order, 1, 0);
    const int wd = (int)l.slot_doubles;
    return io.warm ? launch_k4<ragged_batched_warm_kernel<false>>(ctas, l.threads, smem, stream, a, v.d_lps, order,
                                                                  l.per_cta, wd, io.function)
                   : launch_k4<ragged_batched_kernel<false>>(ctas, l.threads, smem, stream, a, v.d_lps, order,
                                                             l.per_cta, wd);
}

} // namespace spx_launch
