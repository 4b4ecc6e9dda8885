// spx_pick.cu — K1 (pricing) + K2 (ratio test): pick_element(), /root/reference/src/simplex.py:70-141.
//
// One CTA of 1024 threads per pick: every decision of the reference is a
// first-index search or the class-aware ratio scan, restated as order-independent
// reductions (warp shuffle -> shared memory -> warp shuffle), so any tree order
// returns the reference's sequential answer.  The work is O(n + m) against the
// O(n*m) update, and the pivot column is gathered into a contiguous buffer on
// the way so the streaming update never does a strided read.
//
// The same building blocks serve the column-sharded flow: `candidate` is the
// local half of K1 (+ column gather into the all-gather message), `select` is
// the global half of K1 (min key over ranks) + K2 on the winning column.
#include "spx_block.cuh"
#include "spx_launch.cuh"

namespace {

using namespace spx;

constexpr int PICK_THREADS = 1024;
constexpr int MSG_HEADER   = 4;      // doubles: [key_hi, key_lo, r_phase1, reserved]
constexpr int GATHER_BATCH = 8;      // independent loads in flight per thread in the O(n) loops

// ---- peer mailboxes (column-sharded flow over NVLink peer memory) ------------------
// Every rank's candidate message is stored by its owner straight into each peer's mailbox
// (peer_push_kernel, spx_shard.cu) followed by a release-store of the exchange number into the
// peer's flag word; the select kernels acquire-poll their LOCAL flags before reading.  Returns
// false on timeout (a peer died): the caller reports SPX_PEER_TIMEOUT instead of hanging the GPU.
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ bool wait_flags(const unsigned long long *flags, int nranks, unsigned long long seq) {
    bool ok = true;
    if (flags != nullptr && (int)threadIdx.x < nranks) {
        const unsigned long long *f = flags + threadIdx.x;
        const unsigned long long t0 = global_timer_ns();
        for (;;) {
            unsigned long long v;
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
            if (v >= seq) break;
            if (global_timer_ns() - t0 > 20000000000ull) { ok = false; break; }     // 20 s
            __nanosleep(100);
        }
    }
    return __syncthreads_or(ok ? 0 : 1) == 0;
}

// K1 on the columns [0, m_loc) this CTA can see.
//   r1    : phase-1 row (first b < 0, :72-76) or -1
//   cloc  : entering column, local index, or SPX_NONE
//   keyhi : 0 for the reference rule; the order-preserving image of f[cloc] for Dantzig
__device__ void block_entering(const double *__restrict__ A, const double *__restrict__ b,
                               int n, int m_loc, int64_t ld, int rule, const spx_state *st,
                               Scratch &s, int &r1, int &cloc, unsigned long long &keyhi) {
    const int64_t npiv = st->npiv;
    const int sl = (int)(npiv & 1);
    const bool hinted = (st->hint_tag[sl] == npiv);
    keyhi = 0ull;
    const int rb = hinted ? st->hint_bneg[sl] : block_first_index(b, n, IsNeg(), s);
    if (rb != SPX_NONE) {                                              // :79
        r1 = rb;
        cloc = block_first_index(A + (int64_t)rb * ld, m_loc, IsPos(), s);   // :82-85
        return;
    }
    r1 = -1;
    const double *f = A + (int64_t)n * ld;
    if (rule == SPX_RULE_REFERENCE) {                                  // :94-98
        cloc = hinted ? st->hint_fneg[sl] : block_first_index(f, m_loc, IsNeg(), s);
        return;
    }
    // Dantzig: most negative f[j], lowest index on ties
    unsigned long long best = ~0ull;
    for (int j = threadIdx.x; j < m_loc; j += blockDim.x) {
        const double v = f[j];
        if (v < 0.0) { const unsigned long long k = orderable(v); best = k < best ? k : best; }
    }
    best = block_min_u64(best, s);
    if (best == ~0ull) { cloc = SPX_NONE; return; }
    int loc = SPX_NONE;
    for (int j = threadIdx.x; j < m_loc; j += blockDim.x) {
        const double v = f[j];
        if (v < 0.0 && orderable(v) == best) { loc = j; break; }
    }
    cloc = block_min_int(loc, s);
    keyhi = best;
}

// K2 once the entering column is known: gathers the column into colbuf and runs the ratio
// test; every thread returns the same decision.
//   col/stride : where the winning column lives (tableau: stride ld; message: stride 1)
//   r1         : phase-1 row or -1;  cglob : global column index or -1 (none)
//   npiv/cap   : pivots applied to the table being priced / max_pivots
struct Decision { int status; int r; double p; };

// col may point into a peer mailbox that remote GPUs wrote while this kernel was already resident
// (shard_select_kernel / ahead_select_kernel): no __restrict__ and explicit ld.global.cg reads, so the
// compiler can never turn them into non-coherent ld.global.nc loads that the flag acquire does not order.
__device__ Decision block_decide(const double *col, int64_t stride,
                                 const double *__restrict__ b, int n, int r1, int64_t cglob,
                                 int64_t npiv, int64_t cap, double *__restrict__ colbuf, Scratch &s) {
    Decision dec; dec.r = -1; dec.p = 0.0;
    if (cglob < 0) {
        dec.status = (r1 >= 0) ? SPX_INCORRECT : SPX_OPTIMAL;          // :88-89, :101-103
        return dec;
    }
    Ratio q = ratio_identity();
    // GATHER_BATCH independent (strided) loads in flight per thread: the loop is latency-bound
    const int nt = (int)blockDim.x;
    for (int base = 0; base <= n; base += nt * GATHER_BATCH) {
        double a[GATHER_BATCH], bb[GATHER_BATCH];
#pragma unroll
        for (int u = 0; u < GATHER_BATCH; ++u) {
            const int i = base + u * nt + (int)threadIdx.x;
            a[u]  = (i <= n) ? __ldcg(col + (int64_t)i * stride) : 0.0;
            bb[u] = (r1 < 0 && i < n) ? b[i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < GATHER_BATCH; ++u) {
            const int i = base + u * nt + (int)threadIdx.x;
            if (i <= n) {
                colbuf[i] = a[u];
                if (r1 < 0 && i < n) ratio_accumulate(q, i, a[u], bb[u]);   // :111-136
            }
        }
    }
    int r;
    if (r1 >= 0) {
        r = r1;                                                        // :91, no ratio test in phase 1
    } else {
        q = block_ratio_reduce(q, s);
        bool elig_nan = false;
        if (q.elig_row != SPX_NONE) {
            const double v = __ddiv_rn(b[q.elig_row], __ldcg(col + (int64_t)q.elig_row * stride));
            elig_nan = (v != v);
        }
        r = ratio_decide(q, elig_nan);                                 // :138-141
    }
    dec.status = (r < 0) ? SPX_NOCONV : SPX_PIVOT;
    if (dec.status == SPX_PIVOT) {
        dec.r = r;
        dec.p = __ldcg(col + (int64_t)r * stride);
        if (npiv >= cap) dec.status = SPX_CAP;
    }
    return dec;
}

// in-place bookkeeping of the step API (spx_pick / spx_shard_select): the update that follows
// increments npiv and fills the hint slot
__device__ void block_finish(const double *col, int64_t stride,
                             const double *__restrict__ b, int n, int r1, int64_t cglob,
                             spx_state *st, double *__restrict__ colbuf, Scratch &s) {
    const Decision dec = block_decide(col, stride, b, n, r1, cglob, st->npiv, st->max_pivots, colbuf, s);
    __syncthreads();
    if (threadIdx.x == 0) {
        st->status = dec.status;
        st->phase1 = (r1 >= 0) ? 1 : 0;
        if (dec.status == SPX_PIVOT) {
            st->r = dec.r; st->c = cglob; st->p = dec.p;
            const int nslot = (int)((st->npiv + 1) & 1);
            st->slot = nslot;
            st->hint_bneg[nslot] = SPX_NONE;      // the update min-reduces into these
            st->hint_fneg[nslot] = SPX_NONE;
        }
    }
}

__global__ void __launch_bounds__(PICK_THREADS, 1)
pick_kernel(const double *__restrict__ A, const double *__restrict__ b, int n, int m, int64_t ld,
            int rule, int sticky, spx_state *st, double *__restrict__ colbuf) {
    __shared__ Scratch s;
    if (sticky && st->status != SPX_PIVOT) return;
    int r1, cloc; unsigned long long keyhi;
    block_entering(A, b, n, m, ld, rule, st, s, r1, cloc, keyhi);
    const int64_t cglob = (cloc == SPX_NONE) ? -1 : (int64_t)cloc;
    block_finish(A + (cglob < 0 ? 0 : cglob), ld, b, n, r1, cglob, st, colbuf, s);
}

// local half of K1 for one column shard; message = [key_hi, key_lo, r1, 0 | column(n+1)]
__global__ void __launch_bounds__(PICK_THREADS, 1)
shard_candidate_kernel(const double *__restrict__ A, const double *__restrict__ b, int n, int m_loc,
                       int64_t ld, int64_t col0, int rule, int sticky, const spx_state *st,
                       double *__restrict__ msg) {
    __shared__ Scratch s;
    if (sticky && st->status != SPX_PIVOT) return;
    int r1, cloc; unsigned long long keyhi;
    block_entering(A, b, n, m_loc, ld, rule, st, s, r1, cloc, keyhi);
    if (threadIdx.x == 0) {
        unsigned long long *h = reinterpret_cast<unsigned long long *>(msg);
        h[0] = (cloc == SPX_NONE) ? ~0ull : keyhi;
        h[1] = (cloc == SPX_NONE) ? ~0ull : (unsigned long long)(col0 + cloc);
        h[2] = (unsigned long long)(long long)r1;
        h[3] = 0ull;
    }
    if (cloc != SPX_NONE) {
        const double *col = A + cloc;
        const int nt = (int)blockDim.x;
        for (int base = 0; base <= n; base += nt * GATHER_BATCH) {
            double t[GATHER_BATCH];
#pragma unroll
            for (int u = 0; u < GATHER_BATCH; ++u) {
                const int i = base + u * nt + (int)threadIdx.x;
                t[u] = (i <= n) ? col[(int64_t)i * ld] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < GATHER_BATCH; ++u) {
                const int i = base + u * nt + (int)threadIdx.x;
                if (i <= n) msg[MSG_HEADER + i] = t[u];
            }
        }
    }
}

// global half of K1 + K2 from the gathered messages of all ranks
__global__ void __launch_bounds__(PICK_THREADS, 1)
shard_select_kernel(const double *gathered, int nranks, int64_t msg_doubles,
                    const double *__restrict__ b, int n, int sticky, spx_state *st,
                    double *__restrict__ colbuf, const unsigned long long *flags, unsigned long long seq) {
    __shared__ Scratch s;
    if (sticky && st->status != SPX_PIVOT) return;
    if (!wait_flags(flags, nranks, seq)) {
        if (threadIdx.x == 0) st->status = SPX_PEER_TIMEOUT;
        return;
    }
    // every thread scans the (few) headers: lexicographic min of (key_hi, key_lo)
    unsigned long long bh = ~0ull, bl = ~0ull; int win = -1;
    for (int g = 0; g < nranks; ++g) {
        const unsigned long long *h =
            reinterpret_cast<const unsigned long long *>(gathered + (int64_t)g * msg_doubles);
        const unsigned long long kh = h[0], kl = h[1];
        if (kl != ~0ull && (win < 0 || kh < bh || (kh == bh && kl < bl))) { bh = kh; bl = kl; win = g; }
    }
    const int r1 = (int)(long long)reinterpret_cast<const unsigned long long *>(gathered)[2];
    const int64_t cglob = (win < 0) ? -1 : (int64_t)bl;
    const double *col = gathered + (int64_t)(win < 0 ? 0 : win) * msg_doubles + MSG_HEADER;
    block_finish(col, 1, b, n, r1, cglob, st, colbuf, s);
}

// ---- look-ahead pricing ------------------------------------------------------------
// Pivot k+1 is chosen from table k WHILE the streaming update of pivot k runs: every cell the
// choice depends on — the new b column, one new row (f, or the phase-1 row), one new column —
// is O(n + m) work computed here with exactly the update kernel's arithmetic (same pivot_div,
// same operation order), so the decision is the one a pick on the finished table k+1 makes.
// The tableau update then never waits for pricing, and on a column-sharded tableau the
// all-gather of the candidates is off the critical path as well.
constexpr int AHEAD_THREADS = 256;   // fits the slot one retiring update CTA frees

// message layout: [key_hi, key_lo, r1, terminal | new column c' (n+1 cells, f row last)]
__global__ void __launch_bounds__(AHEAD_THREADS, 3)
ahead_candidate_kernel(const double *__restrict__ A, const double *__restrict__ bin,
                       double *__restrict__ bout, int n, int m_loc, int64_t ld, int64_t col0, int rule,
                       const spx_state *__restrict__ st, const double *__restrict__ colbuf,
                       double *__restrict__ msg) {
    __shared__ Scratch s;
    unsigned long long *h = reinterpret_cast<unsigned long long *>(msg);
    if (st->status != SPX_PIVOT) {                       // nothing left to price: select copies the state
        if (threadIdx.x == 0) { h[0] = ~0ull; h[1] = ~0ull; h[2] = ~0ull; h[3] = 1ull; }
        return;
    }
    const int     r  = st->r;
    const int64_t cl = st->c - col0;                     // local index of the current pivot column
    const double  p  = st->p;
    const PivotDiv d = pivot_div_prepare(p);
    const int nt = (int)blockDim.x;

    // 1. the next '-b' column (replicated on every rank), first negative -> phase-1 row (:72-76)
    int bneg = SPX_NONE;
    const double br = bin[r];
    for (int base = 0; base < n; base += nt * GATHER_BATCH) {
        double bi[GATHER_BATCH], ci[GATHER_BATCH];
#pragma unroll
        for (int u = 0; u < GATHER_BATCH; ++u) {
            const int i = base + u * nt + (int)threadIdx.x;
            bi[u] = (i < n) ? bin[i] : 0.0;
            ci[u] = (i < n) ? colbuf[i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < GATHER_BATCH; ++u) {
            const int i = base + u * nt + (int)threadIdx.x;
            if (i < n) {
                const double nb = (i == r) ? pivot_div(-bi[u], d) : cell_update(bi[u], d, br, ci[u]);
                bout[i] = nb;
                if (nb < 0.0) bneg = min(bneg, i);
            }
        }
    }
    const int rb = block_min_int(bneg, s);
    const int r1 = (rb == SPX_NONE) ? -1 : rb;

    // 2. the entering column from one row of the NEXT table: the phase-1 row (:82-85) or f (:94-98)
    const double *rowr = A + (int64_t)r * ld;
    const int     li   = (r1 >= 0) ? r1 : n;             // which row of the table is priced
    const double *rowi = A + (int64_t)li * ld;
    const double  cli  = colbuf[li];
    auto next_cell = [&](int j) -> double {
        if (j == cl) return (li == r) ? pivot_cell_update(p) : pivot_div(cli, d);          // :163, :160
        return (li == r) ? pivot_div(-rowr[j], d) : cell_update(rowi[j], d, rowr[j], cli); // :156, :173-175
    };
    int cloc;
    unsigned long long keyhi = 0ull;
    if (r1 >= 0) {
        cloc = block_first_index_fn(m_loc, next_cell, IsPos(), s);
    } else if (rule == SPX_RULE_REFERENCE) {
        cloc = block_first_index_fn(m_loc, next_cell, IsNeg(), s);
    } else {                                             // Dantzig: most negative, lowest index on ties
        unsigned long long best = ~0ull;
        for (int j = threadIdx.x; j < m_loc; j += nt) {
            const double v = next_cell(j);
            if (v < 0.0) { const unsigned long long k = orderable(v); best = k < best ? k : best; }
        }
        best = block_min_u64(best, s);
        int loc = SPX_NONE;
        if (best != ~0ull)
            for (int j = threadIdx.x; j < m_loc; j += nt) {
                const double v = next_cell(j);
                if (v < 0.0 && orderable(v) == best) { loc = j; break; }
            }
        cloc = block_min_int(loc, s);
        keyhi = best;
    }
    if (threadIdx.x == 0) {
        h[0] = (cloc == SPX_NONE) ? ~0ull : keyhi;
        h[1] = (cloc == SPX_NONE) ? ~0ull : (unsigned long long)(col0 + cloc);
        h[2] = (unsigned long long)(long long)r1;
        h[3] = 0ull;
    }
    if (cloc == SPX_NONE) return;

    // 3. column cloc of the NEXT table (a strided gather of the current one, GATHER_BATCH loads in flight)
    const double rj = rowr[cloc];
    const bool same = (cloc == cl);                      // the column that just left re-enters
    const double *colp = A + cloc;
    double *out = msg + MSG_HEADER;
    for (int base = 0; base <= n; base += nt * GATHER_BATCH) {
        double t[GATHER_BATCH], cc[GATHER_BATCH];
#pragma unroll
        for (int u = 0; u < GATHER_BATCH; ++u) {
            const int i = base + u * nt + (int)threadIdx.x;
            t[u]  = (i <= n && !same) ? colp[(int64_t)i * ld] : 0.0;
            cc[u] = (i <= n) ? colbuf[i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < GATHER_BATCH; ++u) {
            const int i = base + u * nt + (int)threadIdx.x;
            if (i <= n) {
                const double ci = cc[u];
                double v;
                if (same) v = (i == r) ? pivot_cell_update(p) : pivot_div(ci, d);
                else      v = (i == r) ? pivot_div(-rj, d) : cell_update(t[u], d, rj, ci);
                out[i] = v;
            }
        }
    }
}

// global half: min key over the ranks' messages, ratio test on the winning column with the next b,
// next state written to st_next (st_cur is still being read by the running update)
__global__ void __launch_bounds__(AHEAD_THREADS, 3)
ahead_select_kernel(const double *gathered, int nranks, int64_t msg_doubles,
                    const double *__restrict__ bnext, int n, const spx_state *__restrict__ st_cur,
                    spx_state *__restrict__ st_next, double *__restrict__ colbuf_next,
                    const unsigned long long *flags, unsigned long long seq) {
    __shared__ Scratch s;
    if (!wait_flags(flags, nranks, seq)) {
        if (threadIdx.x == 0) { *st_next = *st_cur; st_next->status = SPX_PEER_TIMEOUT; }
        return;
    }
    const unsigned long long *h0 = reinterpret_cast<const unsigned long long *>(gathered);
    if (st_cur->status != SPX_PIVOT || h0[3] != 0ull) {
        if (threadIdx.x == 0) { *st_next = *st_cur; st_next->hint_tag[0] = st_next->hint_tag[1] = -1; }
        return;
    }
    unsigned long long bh = ~0ull, bl = ~0ull; int win = -1;
    for (int g = 0; g < nranks; ++g) {
        const unsigned long long *h =
            reinterpret_cast<const unsigned long long *>(gathered + (int64_t)g * msg_doubles);
        const unsigned long long kh = h[0], kl = h[1];
        if (kl != ~0ull && (win < 0 || kh < bh || (kh == bh && kl < bl))) { bh = kh; bl = kl; win = g; }
    }
    const int r1 = (int)(long long)h0[2];
    const int64_t cglob = (win < 0) ? -1 : (int64_t)bl;
    const double *col = gathered + (int64_t)(win < 0 ? 0 : win) * msg_doubles + MSG_HEADER;
    const int64_t npiv = st_cur->npiv + 1;               // pivots applied to the table being priced
    const int64_t cap  = st_cur->max_pivots;
    const Decision dec = block_decide(col, 1, bnext, n, r1, cglob, npiv, cap, colbuf_next, s);
    if (threadIdx.x == 0) {
        spx_state o;
        o.status = dec.status; o.r = dec.r; o.c = cglob; o.p = dec.p;
        o.npiv = npiv; o.max_pivots = cap; o.phase1 = (r1 >= 0) ? 1 : 0; o.slot = 0;
        o.hint_tag[0] = o.hint_tag[1] = -1;
        o.hint_bneg[0] = o.hint_bneg[1] = SPX_NONE;
        o.hint_fneg[0] = o.hint_fneg[1] = SPX_NONE;
        for (int q = 0; q < 6; ++q) o.reserved[q] = 0;
        *st_next = o;
    }
}

} // namespace

// ---- launchers (called from spx_api.cu) -------------------------------------
namespace spx_launch {

int64_t shard_msg_doubles(int n) {
    int64_t d = MSG_HEADER + (int64_t)n + 1;
    return (d + 15) / 16 * 16;
}

cudaError_t pick(const double *A, const double *b, int n, int m, int64_t ld, int rule, int sticky,
                 spx_state *st, double *colbuf, cudaStream_t stream) {
    pick_kernel<<<1, PICK_THREADS, 0, stream>>>(A, b, n, m, ld, rule, sticky, st, colbuf);
    spx_host::count_launch();
    return cudaGetLastError();
}

cudaError_t shard_candidate(const double *A, const double *b, int n, int m_loc, int64_t ld,
                            int64_t col0, int rule, int sticky, const spx_state *st, double *msg,
                            cudaStream_t stream) {
    shard_candidate_kernel<<<1, PICK_THREADS, 0, stream>>>(A, b, n, m_loc, ld, col0, rule, sticky,
                                                           st, msg);
    spx_host::count_launch();
    return cudaGetLastError();
}

cudaError_t shard_select(const double *gathered, int nranks, const double *b, int n, int sticky,
                         spx_state *st, double *colbuf, const unsigned long long *flags,
                         unsigned long long seq, cudaStream_t stream) {
    shard_select_kernel<<<1, PICK_THREADS, 0, stream>>>(gathered, nranks, shard_msg_doubles(n), b,
                                                        n, sticky, st, colbuf, flags, seq);
    spx_host::count_launch();
    return cudaGetLastError();
}

cudaError_t ahead_candidate(const double *A, const double *bin, double *bout, int n, int m_loc,
                            int64_t ld, int64_t col0, int rule, const spx_state *st,
                            const double *colbuf, double *msg, cudaStream_t stream) {
    ahead_candidate_kernel<<<1, AHEAD_THREADS, 0, stream>>>(A, bin, bout, n, m_loc, ld, col0, rule, st,
                                                            colbuf, msg);
    spx_host::count_launch();
    return cudaGetLastError();
}

cudaError_t ahead_select(const double *gathered, int nranks, const double *bnext, int n,
                         const spx_state *st_cur, spx_state *st_next, double *colbuf_next,
                         const unsigned long long *flags, unsigned long long seq, cudaStream_t stream) {
    ahead_select_kernel<<<1, AHEAD_THREADS, 0, stream>>>(gathered, nranks, shard_msg_doubles(n), bnext, n,
                                                         st_cur, st_next, colbuf_next, flags, seq);
    spx_host::count_launch();
    return cudaGetLastError();
}

} // namespace spx_launch
