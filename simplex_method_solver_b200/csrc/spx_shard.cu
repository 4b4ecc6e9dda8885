// spx_shard.cu — the column-sharded pivot loop over NVLink peer memory, one process per GPU.
//
// The reference has no multi-device path (SURVEY.md §2); this is the B200-native way the pivot
// loop of /root/reference/src/simplex.py:179-199 shards for a tableau larger than one GPU wants
// to stream: rank g owns a block of columns, b / labels / state are replicated, and the only
// exchange per pivot is each rank's candidate message [key | its entering column] (128 KB at
// n = 16384).  The exchange is not a library collective: every rank STORES its message into each
// peer's mailbox through NVLink (peer_push_kernel: 128-bit stores to peer-mapped addresses, one CTA
// per destination), then release-stores the exchange number into the peer's flag word; the select
// kernel of the destination acquire-polls its LOCAL flags (wait_flags, spx_pick.cu).  No NCCL call,
// no host round trip and — in look-ahead mode — no exchange latency on the critical path: pivot
// k+1 is priced on the side stream while update k streams on the main stream.
//
// Mailbox of one rank (spx_mailbox_bytes):  gathered[2][nranks][msg]  |  flags[2][nranks]
// Two parities: a fast rank may already push exchange s+1 while a slow rank still reads
// exchange s; it cannot reach s+2 before every rank has finished reading s (its own select(s+1)
// needs everyone's push(s+1), which each rank issues after its select(s)).
#include <cstring>
#include <new>

#include "spx_launch.cuh"

namespace {

constexpr int MAX_RANKS = 16;
constexpr int PUSH_THREADS = 256;

struct PeerBoxes { unsigned char *box[MAX_RANKS]; };

inline int64_t align128(int64_t v) { return (v + 127) / 128 * 128; }
inline int64_t gathered_bytes(int n, int nranks) {
    return align128(2LL * nranks * spx_launch::shard_msg_doubles(n) * 8);
}

// CTA g stores this rank's message into rank g's mailbox, then publishes the exchange number
__global__ void __launch_bounds__(PUSH_THREADS)
peer_push_kernel(const double *__restrict__ send, int64_t msg_doubles, int rank, int nranks, int parity,
                 unsigned long long seq, int64_t flags_offset, PeerBoxes peers) {
    const int g = blockIdx.x;
    unsigned char *box = peers.box[g];
    double2 *dst = reinterpret_cast<double2 *>(box) + ((int64_t)parity * nranks + rank) * (msg_doubles / 2);
    const double2 *src = reinterpret_cast<const double2 *>(send);
    const int64_t count = msg_doubles / 2;                         // msg_doubles is a multiple of 16
    for (int64_t base = 0; base < count; base += PUSH_THREADS * 4) {
        double2 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t k = base + u * PUSH_THREADS + threadIdx.x;
            if (k < count) v[u] = src[k];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t k = base + u * PUSH_THREADS + threadIdx.x;
            if (k < count) dst[k] = v[u];
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long *flag =
            reinterpret_cast<unsigned long long *>(box + flags_offset) + (int64_t)parity * nranks + rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(flag), "l"(seq) : "memory");
    }
}

} // namespace

struct spx_shard {
    int rank, nranks, n, m_loc, rule;
    int64_t ld, col0, msgd, flags_offset;
    double *A[2], *b[2];
    spx_state *S[2];
    double *C[2];
    int32_t *rowlab, *collab, *trace;
    double *send;
    PeerBoxes peers;
    unsigned char *mybox;
    int si;                    // which state / colbuf holds the decision for the current table
    bool priced;
    int64_t enqueued;          // pivots enqueued since load (parity of the table buffers)
    unsigned long long seq;    // exchanges issued so far
    cudaStream_t side;
    cudaEvent_t fork, join;
};

using spx_host::check;
using spx_host::set_error;

#define SPX_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            set_error(__VA_ARGS__);       \
            return -2;                    \
        }                                 \
    } while (0)

static cudaError_t exchange(spx_shard *h, cudaStream_t s, unsigned long long *seq_out, int *parity_out) {
    const unsigned long long seq = ++h->seq;
    const int parity = (int)(seq & 1ull);
    peer_push_kernel<<<h->nranks, PUSH_THREADS, 0, s>>>(h->send, h->msgd, h->rank, h->nranks, parity, seq,
                                                        h->flags_offset, h->peers);
    spx_host::count_launch();
    *seq_out = seq;
    *parity_out = parity;
    return cudaGetLastError();
}

static inline const double *gathered_of(const spx_shard *h, int parity) {
    return reinterpret_cast<const double *>(h->mybox) + (int64_t)parity * h->nranks * h->msgd;
}
static inline const unsigned long long *flags_of(const spx_shard *h, int parity) {
    return reinterpret_cast<const unsigned long long *>(h->mybox + h->flags_offset) + (int64_t)parity * h->nranks;
}

extern "C" {

// ---- peer memory plumbing (cudaMalloc'ed so that it can be exported over CUDA IPC) -----------
int spx_device_alloc(void **d_ptr, int64_t bytes) {
    SPX_REQUIRE(d_ptr && bytes > 0, "spx_device_alloc: bad arguments");
    if (check(cudaMalloc(d_ptr, (size_t)bytes), "cudaMalloc")) return -1;
    if (check(cudaMemset(*d_ptr, 0, (size_t)bytes), "cudaMemset")) return -1;
    return check(cudaDeviceSynchronize(), "sync");
}

int spx_device_free(void *d_ptr) { return check(cudaFree(d_ptr), "cudaFree"); }

int spx_ipc_handle_bytes(void) { return (int)sizeof(cudaIpcMemHandle_t); }

int spx_ipc_export(void *d_ptr, void *handle_out) {
    SPX_REQUIRE(d_ptr && handle_out, "spx_ipc_export: null pointer");
    cudaIpcMemHandle_t hnd;
    if (check(cudaIpcGetMemHandle(&hnd, d_ptr), "cudaIpcGetMemHandle")) return -1;
    memcpy(handle_out, &hnd, sizeof(hnd));
    return 0;
}

int spx_ipc_import(const void *handle, void **d_ptr) {
    SPX_REQUIRE(handle && d_ptr, "spx_ipc_import: null pointer");
    cudaIpcMemHandle_t hnd;
    memcpy(&hnd, handle, sizeof(hnd));
    return check(cudaIpcOpenMemHandle(d_ptr, hnd, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle");
}

int spx_ipc_close(void *d_ptr) { return check(cudaIpcCloseMemHandle(d_ptr), "cudaIpcCloseMemHandle"); }

int64_t spx_mailbox_bytes(int32_t n, int32_t nranks) {
    if (n < 1 || nranks < 1 || nranks > MAX_RANKS) return -1;
    return gathered_bytes(n, nranks) + align128(2LL * nranks * 8);
}

// one exchange step on its own (tests emulate several ranks in one process with these)
int spx_peer_push(const double *d_send, int32_t n, int32_t rank, int32_t nranks, int32_t parity,
                  uint64_t seq, void *const *mailboxes, void *stream) {
    SPX_REQUIRE(d_send && mailboxes && n >= 1 && nranks >= 1 && nranks <= MAX_RANKS && rank >= 0 && rank < nranks &&
                (parity == 0 || parity == 1), "spx_peer_push: bad arguments");
    PeerBoxes pb{};
    for (int g = 0; g < nranks; ++g) {
        SPX_REQUIRE(mailboxes[g], "spx_peer_push: null mailbox %d", g);
        pb.box[g] = static_cast<unsigned char *>(mailboxes[g]);
    }
    peer_push_kernel<<<nranks, PUSH_THREADS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        d_send, spx_launch::shard_msg_doubles(n), rank, nranks, parity, seq, gathered_bytes(n, nranks), pb);
    spx_host::count_launch();
    return check(cudaGetLastError(), "push launch");
}

// ---- the handle ---------------------------------------------------------------------------
int spx_shard_open(spx_shard **out, int32_t rank, int32_t nranks, int32_t n, int32_t m_loc, int64_t ld_loc,
                   int64_t col0, int32_t rule, double *d_A0, double *d_A1, double *d_b0, double *d_b1,
                   spx_state *d_state2, double *d_colbuf2, int32_t *d_rowlab, int32_t *d_collab,
                   int32_t *d_trace, double *d_send, void *const *mailboxes) {
    SPX_REQUIRE(out && d_A0 && d_A1 && d_b0 && d_b1 && d_state2 && d_colbuf2 && d_rowlab && d_collab && d_send &&
                mailboxes, "spx_shard_open: null pointer");
    SPX_REQUIRE(nranks >= 1 && nranks <= MAX_RANKS && rank >= 0 && rank < nranks, "spx_shard_open: bad rank %d/%d",
                rank, nranks);
    SPX_REQUIRE(n >= 1 && m_loc >= 0 && ld_loc >= 16 && ld_loc % 16 == 0 && ld_loc >= m_loc && col0 >= 0,
                "spx_shard_open: bad shape");
    SPX_REQUIRE(rule != SPX_RULE_DEVEX && rule != SPX_RULE_DANTZIG_BLAND, "spx_shard_open: rule %s is a rule of the "
                "batched entries only (spx_solve_batched, spx_solve_batched_cluster, spx_solve_batched_global, "
                "spx_solve_batched_ragged, spx_warm_solve_batched, spx_warm_solve_ragged)",
                rule == SPX_RULE_DEVEX ? "SPX_RULE_DEVEX" : "SPX_RULE_DANTZIG_BLAND");
    SPX_REQUIRE(rule == SPX_RULE_REFERENCE || rule == SPX_RULE_DANTZIG, "spx_shard_open: unknown rule %d", rule);
    spx_shard *h = new (std::nothrow) spx_shard();
    SPX_REQUIRE(h, "spx_shard_open: out of host memory");
    h->rank = rank; h->nranks = nranks; h->n = n; h->m_loc = m_loc; h->rule = rule;
    h->ld = ld_loc; h->col0 = col0;
    h->msgd = spx_launch::shard_msg_doubles(n);
    h->flags_offset = gathered_bytes(n, nranks);
    h->A[0] = d_A0; h->A[1] = d_A1; h->b[0] = d_b0; h->b[1] = d_b1;
    h->S[0] = d_state2; h->S[1] = d_state2 + 1;
    h->C[0] = d_colbuf2; h->C[1] = d_colbuf2 + spx_launch::colbuf_doubles(n);
    h->rowlab = d_rowlab; h->collab = d_collab; h->trace = d_trace; h->send = d_send;
    for (int g = 0; g < nranks; ++g) {
        if (!mailboxes[g]) { delete h; set_error("spx_shard_open: null mailbox %d", g); return -2; }
        h->peers.box[g] = static_cast<unsigned char *>(mailboxes[g]);
    }
    h->mybox = h->peers.box[rank];
    h->si = 0; h->priced = false; h->enqueued = 0; h->seq = 0;
    int lo = 0, hi = 0;
    if (check(cudaDeviceGetStreamPriorityRange(&lo, &hi), "priority range") ||
        check(cudaStreamCreateWithPriority(&h->side, cudaStreamNonBlocking, hi), "side stream") ||
        check(cudaEventCreateWithFlags(&h->fork, cudaEventDisableTiming), "event") ||
        check(cudaEventCreateWithFlags(&h->join, cudaEventDisableTiming), "event")) {
        delete h;
        return -1;
    }
    *out = h;
    return 0;
}

int spx_shard_close(spx_shard *h) {
    if (!h) return 0;
    cudaStreamSynchronize(h->side);
    cudaEventDestroy(h->fork);
    cudaEventDestroy(h->join);
    cudaStreamDestroy(h->side);
    delete h;
    return 0;
}

// The state in S[0] was (re)initialised by spx_init_state and table 0 imported: start over.
int spx_shard_reset(spx_shard *h) {
    SPX_REQUIRE(h, "spx_shard_reset: null handle");
    h->si = 0; h->priced = false; h->enqueued = 0;
    return 0;                                   // seq keeps counting: mailbox flags are monotonic
}

// Enqueue `pivots` look-ahead pivots (asynchronous).  Every rank must enqueue the same count.
int spx_shard_enqueue(spx_shard *h, int64_t pivots, void *stream) {
    SPX_REQUIRE(h && pivots >= 0, "spx_shard_enqueue: bad arguments");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    unsigned long long seq; int par;
    if (!h->priced && pivots > 0) {
        // the decision for the current table: classic local half -> push -> global half
        const int cur = (int)(h->enqueued & 1);
        if (check(spx_launch::shard_candidate(h->A[cur], h->b[cur], h->n, h->m_loc, h->ld, h->col0, h->rule, 1,
                                              h->S[h->si], h->send, s), "candidate launch")) return -1;
        if (check(exchange(h, s, &seq, &par), "push launch")) return -1;
        if (check(spx_launch::shard_select(gathered_of(h, par), h->nranks, h->b[cur], h->n, 1, h->S[h->si],
                                           h->C[h->si], flags_of(h, par), seq, s), "select launch")) return -1;
        h->priced = true;
    }
    for (int64_t q = 0; q < pivots; ++q) {
        const int cur = (int)(h->enqueued & 1), si = h->si;
        // side stream: price pivot k+1 from table k (next b, candidate, push, select -> S[si^1], C[si^1])
        if (check(cudaEventRecord(h->fork, s), "fork")) return -1;
        if (check(cudaStreamWaitEvent(h->side, h->fork, 0), "fork wait")) return -1;
        if (check(spx_launch::ahead_candidate(h->A[cur], h->b[cur], h->b[cur ^ 1], h->n, h->m_loc, h->ld, h->col0,
                                              h->rule, h->S[si], h->C[si], h->send, h->side), "candidate launch")) return -1;
        if (check(exchange(h, h->side, &seq, &par), "push launch")) return -1;
        if (check(spx_launch::ahead_select(gathered_of(h, par), h->nranks, h->b[cur ^ 1], h->n, h->S[si], h->S[si ^ 1],
                                           h->C[si ^ 1], flags_of(h, par), seq, h->side), "select launch")) return -1;
        if (check(cudaEventRecord(h->join, h->side), "join")) return -1;
        // main stream: the streaming update of pivot k on this rank's columns
        if (check(spx_launch::update(h->A[cur], h->A[cur ^ 1], h->b[cur], h->b[cur ^ 1], h->n, h->m_loc, h->ld,
                                     h->col0, h->S[si], h->C[si], h->rowlab, h->collab, h->trace, 1, s),
                  "update launch")) return -1;
        if (check(cudaStreamWaitEvent(s, h->join, 0), "join wait")) return -1;
        h->si ^= 1;
        ++h->enqueued;
    }
    return 0;
}

// Synchronise and read the current (already priced) state; re-derives the table parity from the
// pivots actually applied, so enqueueing past a terminal status is harmless.
int spx_shard_read(spx_shard *h, spx_state *h_state, int32_t *cur_buffer, void *stream) {
    SPX_REQUIRE(h && h_state, "spx_shard_read: bad arguments");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (check(cudaMemcpyAsync(h_state, h->S[h->si], sizeof(spx_state), cudaMemcpyDeviceToHost, s), "read state")) return -1;
    if (check(cudaStreamSynchronize(s), "sync")) return -1;
    if (h_state->status != SPX_PIVOT) h->enqueued = h_state->npiv;
    if (cur_buffer) *cur_buffer = (int32_t)(h->enqueued & 1);
    return 0;
}

} // extern "C"
