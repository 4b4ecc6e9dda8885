// spx_api.cu — the extern "C" boundary of libspx_b200.so (see include/spx_b200.h).
// Plain pointers and sizes only; no torch types.  Every entry validates its
// arguments, launches on the caller's stream and reports failures through
// spx_last_error().
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <vector>

#include "spx_launch.cuh"

namespace spx_host {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check(cudaError_t e, const char *what) {
    if (e == cudaSuccess) return 0;
    set_error("%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    return -1;
}

// puts printf-style text in front of the current error message
void prefix_error(const char *fmt, ...) {
    char msg[sizeof(g_err)];
    std::memcpy(msg, g_err, sizeof(msg));
    va_list ap;
    va_start(ap, fmt);
    const int k = vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    if (k >= 0 && k < (int)sizeof(g_err)) snprintf(g_err + k, sizeof(g_err) - k, "%s", msg);
}

void count_launch(int k) { g_launches.fetch_add(k, std::memory_order_relaxed); }

} // namespace spx_host

using spx_host::check;
using spx_host::prefix_error;
using spx_host::set_error;

#define SPX_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            set_error(__VA_ARGS__);       \
            return -2;                    \
        }                                 \
    } while (0)

static inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

// ---- batched routing: which kernel takes an n x m LP under an engine code (K4, K7, K8) ------------------------
namespace {

bool known_engine(int engine) {
    return (engine >= SPX_ENGINE_AUTO && engine <= SPX_ENGINE_CLUSTER) || engine == SPX_ENGINE_GLOBAL ||
           engine == SPX_ENGINE_AUTO_GLOBAL;
}

// The capacity a one-cluster solver's footprint test `fits` (cluster_fits, global_fits) denies an n x m LP.  A
// footprint grows with n and m and shrinks as S grows, so the limits are those of S = 16, found by bisection.
void capacity_text(char *buf, size_t len, int64_t n, int64_t m, bool (*fits)(int64_t, int64_t, int)) {
    auto last = [](int64_t lo, int64_t hi, auto ok) {     // the largest v in [lo, hi) with ok(v), given ok(lo), !ok(hi)
        while (hi - lo > 1) {
            const int64_t mid = lo + (hi - lo) / 2;
            (ok(mid) ? lo : hi) = mid;
        }
        return lo;
    };
    const int64_t cols = last(1, (int64_t)INT32_MAX + 1, [&](int64_t v) { return fits(1, v, 16); });
    if (m > cols) {
        snprintf(buf, len, "capacity: at most %lld columns fit one cluster", (long long)cols);
        return;
    }
    snprintf(buf, len, "capacity: at m = %lld one cluster of 16 CTAs holds at most n = %lld rows, and at most %lld "
             "columns fit one cluster", (long long)m, (long long)last(1, n, [&](int64_t v) { return fits(v, m, 16); }),
             (long long)cols);
}

// Where one LP runs: the kernel, its cluster size and its dynamic shared memory per CTA at that size.
struct Route {
    int     kernel;     // spx::RaggedKernel: RAGGED_WARP or RAGGED_CTA (K4), RAGGED_CLUSTER (K7), RAGGED_GLOBAL (K8)
    int     S;          // K7: the cluster size; K8: S_min, or the forced size; K4: 1
    int64_t bytes;      // at S; K4 warp mode: the LP's slot
};

// The one routing rule of the batched engines, for an n x m LP (n, m >= 1) under a known engine code, with
// `forced` the cluster size SPX_OPT_CLUSTER_SIZE forces (0: none).  AUTO: K4 when batched_fits, else K7; SMEM,
// CLUSTER, GLOBAL: that engine; AUTO_GLOBAL: AUTO, with K8 above K7's capacity.  False, with the error message
// naming the capacity the LP exceeds, when that engine cannot take it.
bool route_lp(int n, int m, int engine, int forced, Route *r) {
    using namespace spx;
    const int64_t cells = spx_cells(n, m);
    const bool k4 = engine == SPX_ENGINE_SMEM ||
                    ((engine == SPX_ENGINE_AUTO || engine == SPX_ENGINE_AUTO_GLOBAL) && spx_launch::batched_fits(n, m));
    const bool k8 = engine == SPX_ENGINE_GLOBAL ||
                    (engine == SPX_ENGINE_AUTO_GLOBAL && !k4 && spx_launch::cluster_size(n, m) == 0);
    char cap[192];
    r->S = 1;
    if (k4) {
        r->bytes = spx_launch::ragged_batched_bytes(n, m, &r->kernel);
        if (r->bytes > 0) return true;
        if (cells > spx_launch::batched_max_cells())
            set_error("%lld cells per LP exceed the shared-memory resident limit %lld", (long long)cells,
                      (long long)spx_launch::batched_max_cells());
        else
            set_error("a %d x %d LP (%lld cells) does not fit the shared memory of one CTA", n, m, (long long)cells);
        return false;
    }
    if (k8) {
        const int smin = spx_launch::global_min_cluster_size(n, m);
        if (smin == 0) {
            capacity_text(cap, sizeof(cap), n, m, spx_launch::global_fits);
            set_error("a %d x %d LP exceeds the shared memory of one cluster (16 CTAs of 227 KB: 8*(2m+1+R) + 4*(R+Q) "
                      "<= 230400 bytes with R = ceil(n/S), Q = ceil(m/S), S <= 16); %s", n, m, cap);
            return false;
        }
        if (forced && smin > forced) {
            set_error("a %d x %d LP does not fit a cluster of SPX_OPT_CLUSTER_SIZE = %d CTAs (8*(2m+1+R) + 4*(R+Q) "
                      "<= 230400 bytes; at least %d CTAs)", n, m, forced, smin);
            return false;
        }
        r->kernel = RAGGED_GLOBAL;
        r->S = forced ? forced : smin;
        r->bytes = spx_launch::ragged_global_bytes(n, m, r->S);
        return true;
    }
    if (spx_launch::cluster_size(n, m) == 0) {
        capacity_text(cap, sizeof(cap), n, m, spx_launch::cluster_fits);
        set_error("a %d x %d LP exceeds one cluster (16 CTAs of 227 KB shared memory: 8*(R*(m+2)+2m+1) + 4*(R+Q) "
                  "<= 230400 bytes with R = ceil(n/16), Q = ceil(m/16)); %s", n, m, cap);
        return false;
    }
    if (forced && !spx_launch::cluster_fits(n, m, forced)) {
        set_error("a %d x %d LP does not fit a cluster of SPX_OPT_CLUSTER_SIZE = %d CTAs", n, m, forced);
        return false;
    }
    r->kernel = RAGGED_CLUSTER;
    r->S = forced ? forced : spx_launch::cluster_size(n, m);
    r->bytes = spx_launch::ragged_cluster_bytes(n, m, r->S);
    return true;
}

int forced_cluster_size() { return (int)spx_launch::get_option(SPX_OPT_CLUSTER_SIZE); }

// the result of a K7 or K8 launch, with the refusal of a device that cannot co-schedule one cluster spelled out
int check_cluster_launch(cudaError_t e, const char *who, int S, int64_t smem) {
    if (e != cudaErrorInvalidClusterSize) return check(e, who);
    set_error("%s: the device cannot co-schedule one cluster of S = %d CTAs with %lld bytes of shared memory each "
              "(cudaOccupancyMaxActiveClusters = 0)", who, S, (long long)smem);
    return -1;
}

// One uniform solve (io.warm == false) or resume (io.warm == true) on the engine route_lp gives `engine`: the body of
// spx_solve_batched, spx_solve_batched_cluster, spx_solve_batched_global and spx_warm_solve_batched.  K4 reads no
// forced cluster size; K7 and K8 check the grid limit, and K8 launches at spx_global_cluster_size.
int solve_uniform(const char *who, int engine, int64_t B, int32_t n, int32_t m, int32_t max_pivots,
                  const spx::BatchIO &io, void *stream) {
    SPX_REQUIRE(known_engine(engine), "%s: unknown engine %d", who, engine);
    SPX_REQUIRE(B >= 0 && n >= 1 && m >= 1 && max_pivots >= 0, "%s: bad arguments", who);
    SPX_REQUIRE(B == 0 || (io.T && io.status && io.npiv), "%s: null T/status/npiv", who);
    SPX_REQUIRE(!io.warm || B == 0 || (io.rowlab && io.collab), "%s: null rowlab/collab (the labels to resume from)",
                who);
    SPX_REQUIRE(!io.warm || B == 0 || !io.obj || io.function, "%s: null function with obj", who);
    SPX_REQUIRE(io.rule == SPX_RULE_REFERENCE || io.rule == SPX_RULE_DANTZIG, "%s: unknown rule %d", who, io.rule);
    Route r;
    if (!route_lp(n, m, engine, forced_cluster_size(), &r)) {
        prefix_error("%s: ", who);
        return -2;
    }
    cudaStream_t s = as_stream(stream);
    if (r.kernel == spx::RAGGED_WARP || r.kernel == spx::RAGGED_CTA)
        return check(spx_launch::solve_batched(B, n, m, max_pivots, io, s), "batched launch");
    // K8: a default S above S_min is only chosen when all B clusters are co-resident, far below the grid limit
    SPX_REQUIRE(B <= INT32_MAX / r.S, "%s: B = %lld LPs x S = %d CTAs exceed one grid", who, (long long)B, r.S);
    if (r.kernel == spx::RAGGED_CLUSTER)
        return check_cluster_launch(spx_launch::solve_batched_cluster(B, n, m, r.S, max_pivots, io, s), who, r.S,
                                    r.bytes);
    if (B == 0) return 0;
    int S = 0;
    char what[96];
    snprintf(what, sizeof(what), "%s: occupancy", who);
    if (check(spx_launch::global_cluster_size(n, m, B, &S), what)) return -1;
    return check_cluster_launch(spx_launch::solve_batched_global(B, n, m, S, max_pivots, io, s), who, S,
                                spx_launch::ragged_global_bytes(n, m, S));
}

} // namespace

extern "C" {

int spx_version(void) { return SPX_ABI_VERSION; }

const char *spx_last_error(void) { return spx_host::g_err; }

int64_t spx_ld(int64_t m) {
    int64_t ld = (m + 15) / 16 * 16;
    return ld < 16 ? 16 : ld;
}

int64_t spx_cells(int32_t n, int32_t m) { return (int64_t)n * (m + 1) + m; }

int64_t spx_colbuf_doubles(int32_t n) { return spx_launch::colbuf_doubles(n); }

int spx_state_bytes(void) { return (int)sizeof(spx_state); }

int spx_device_info(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor) {
    int dev = 0;
    if (check(cudaGetDevice(&dev), "cudaGetDevice")) return -1;
    int sms = 0, maj = 0, min = 0;
    if (check(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev), "attr")) return -1;
    if (check(cudaDeviceGetAttribute(&maj, cudaDevAttrComputeCapabilityMajor, dev), "attr")) return -1;
    if (check(cudaDeviceGetAttribute(&min, cudaDevAttrComputeCapabilityMinor, dev), "attr")) return -1;
    if (sm_count) *sm_count = sms;
    if (cc_major) *cc_major = maj;
    if (cc_minor) *cc_minor = min;
    return 0;
}

int64_t spx_launch_count(int reset) {
    long long v = spx_host::g_launches.load(std::memory_order_relaxed);
    if (reset) spx_host::g_launches.store(0, std::memory_order_relaxed);
    return v;
}

int spx_set_option(int32_t option, int64_t value) {
    if (spx_launch::set_option(option, value) != 0) {
        set_error("spx_set_option: bad option %d / value %lld", option, (long long)value);
        return -2;
    }
    return 0;
}

int64_t spx_get_option(int32_t option) { return spx_launch::get_option(option); }

int spx_selftest_division(const double *d_a, const double *d_p, int64_t count, int64_t np,
                          uint64_t *h_mismatches, double *h_first_bad, void *stream) {
    SPX_REQUIRE(d_a && d_p && h_mismatches && count >= 0 && np >= 1, "spx_selftest_division: bad arguments");
    cudaStream_t s = as_stream(stream);
    unsigned long long *d_cnt = nullptr;
    double *d_bad = nullptr;
    if (check(cudaMalloc(&d_cnt, sizeof(*d_cnt)), "cudaMalloc")) return -1;
    if (check(cudaMalloc(&d_bad, 2 * sizeof(double)), "cudaMalloc")) { cudaFree(d_cnt); return -1; }
    int rc = 0;
    double bad[2] = {0.0, 0.0};
    unsigned long long cnt = 0;
    if (check(cudaMemsetAsync(d_cnt, 0, sizeof(*d_cnt), s), "memset") ||
        check(cudaMemsetAsync(d_bad, 0, 2 * sizeof(double), s), "memset") ||
        check(spx_launch::selftest_division(d_a, d_p, count, np, d_cnt, d_bad, s), "selftest launch") ||
        check(cudaMemcpyAsync(&cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, s), "read") ||
        check(cudaMemcpyAsync(bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost, s), "read") ||
        check(cudaStreamSynchronize(s), "sync"))
        rc = -1;
    cudaFree(d_cnt);
    cudaFree(d_bad);
    *h_mismatches = cnt;
    if (h_first_bad) { h_first_bad[0] = bad[0]; h_first_bad[1] = bad[1]; }
    return rc;
}

int spx_selftest_lazy_guard(const double *d_t0, const double *d_p, const double *d_rj, const double *d_ci,
                            int32_t levels, int64_t count, double *d_out_lazy, double *d_out_ref,
                            uint64_t *h_redo, void *stream) {
    SPX_REQUIRE(d_t0 && d_p && d_rj && d_ci && d_out_lazy && d_out_ref && h_redo && count >= 0 && levels >= 1 &&
                levels <= spx_launch::fuse_max(), "spx_selftest_lazy_guard: bad arguments");
    cudaStream_t s = as_stream(stream);
    unsigned long long *d_cnt = nullptr, cnt = 0;
    if (check(cudaMalloc(&d_cnt, sizeof(*d_cnt)), "cudaMalloc")) return -1;
    int rc = 0;
    if (check(cudaMemsetAsync(d_cnt, 0, sizeof(*d_cnt), s), "memset") ||
        check(spx_launch::lazy_guard_selftest(d_t0, d_p, d_rj, d_ci, levels, count, d_out_lazy, d_out_ref, d_cnt, s),
              "selftest launch") ||
        check(cudaMemcpyAsync(&cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, s), "read") ||
        check(cudaStreamSynchronize(s), "sync"))
        rc = -1;
    cudaFree(d_cnt);
    *h_redo = cnt;
    return rc;
}

// ---- layout conversion ---------------------------------------------------------
int spx_import_shard(const double *src_rows, const double *src_function, double *d_A, double *d_b,
                     int32_t n, int32_t m, int64_t col0, int32_t m_loc, int64_t ld_loc, void *stream) {
    SPX_REQUIRE(src_rows && (src_function || m_loc == 0) && d_A, "spx_import_shard: null pointer");
    // m == 0 is a packed block of a rank that owns no columns: rows of ONE cell, the b column (pitch 8 bytes)
    SPX_REQUIRE(n >= 0 && (m >= 1 || (m == 0 && m_loc == 0)) && m_loc >= 0 && col0 >= 0 && col0 + m_loc <= m,
                "spx_import_shard: bad shape n=%d m=%d col0=%lld m_loc=%d", n, m, (long long)col0, m_loc);
    SPX_REQUIRE(ld_loc >= m_loc && ld_loc % 16 == 0, "spx_import_shard: ld=%lld must be a multiple of 16 >= m_loc",
                (long long)ld_loc);
    cudaStream_t s = as_stream(stream);
    const size_t spitch = (size_t)(m + 1) * sizeof(double);
    const size_t dpitch = (size_t)ld_loc * sizeof(double);
    if (m_loc > 0 && n > 0)
        if (check(cudaMemcpy2DAsync(d_A, dpitch, src_rows + col0, spitch, (size_t)m_loc * sizeof(double),
                                    (size_t)n, cudaMemcpyDefault, s), "import body")) return -1;
    if (m_loc > 0)   // the f row has m cells (simplex.py:39)
        if (check(cudaMemcpyAsync(d_A + (size_t)n * ld_loc, src_function + col0,
                                  (size_t)m_loc * sizeof(double), cudaMemcpyDefault, s), "import f row")) return -1;
    if (ld_loc > m_loc)
        if (check(cudaMemset2DAsync(d_A + m_loc, dpitch, 0, (size_t)(ld_loc - m_loc) * sizeof(double),
                                    (size_t)n + 1, s), "zero padding")) return -1;
    if (d_b && n > 0)
        if (check(cudaMemcpy2DAsync(d_b, sizeof(double), src_rows + m, spitch, sizeof(double), (size_t)n,
                                    cudaMemcpyDefault, s), "import b")) return -1;
    return 0;
}

int spx_import_table(const double *src_rows, const double *src_function, double *d_A, double *d_b,
                     int32_t n, int32_t m, int64_t ld, void *stream) {
    SPX_REQUIRE(d_b, "spx_import_table: null d_b");
    return spx_import_shard(src_rows, src_function, d_A, d_b, n, m, 0, m, ld, stream);
}

int spx_export_table(const double *d_A, const double *d_b, double *dst_rows, double *dst_function,
                     int32_t n, int32_t m, int64_t ld, void *stream) {
    SPX_REQUIRE(d_A && d_b && dst_rows && dst_function, "spx_export_table: null pointer");
    SPX_REQUIRE(n >= 0 && m >= 1 && ld >= m, "spx_export_table: bad shape");
    cudaStream_t s = as_stream(stream);
    const size_t dpitch = (size_t)(m + 1) * sizeof(double);
    const size_t spitch = (size_t)ld * sizeof(double);
    if (n > 0) {
        if (check(cudaMemcpy2DAsync(dst_rows, dpitch, d_A, spitch, (size_t)m * sizeof(double), (size_t)n,
                                    cudaMemcpyDefault, s), "export body")) return -1;
        if (check(cudaMemcpy2DAsync(dst_rows + m, dpitch, d_b, sizeof(double), sizeof(double), (size_t)n,
                                    cudaMemcpyDefault, s), "export b")) return -1;
    }
    if (check(cudaMemcpyAsync(dst_function, d_A + (size_t)n * ld,
                              (size_t)m * sizeof(double), cudaMemcpyDefault, s), "export f row")) return -1;
    return 0;
}

int spx_init_state(spx_state *d_state, int32_t *d_rowlab, int32_t *d_collab, int32_t n, int32_t m,
                   int64_t max_pivots, void *stream) {
    SPX_REQUIRE(d_state && d_rowlab && d_collab, "spx_init_state: null pointer");
    SPX_REQUIRE(n >= 0 && m >= 1 && max_pivots >= 0, "spx_init_state: bad arguments");
    return check(spx_launch::init_state(d_state, d_rowlab, d_collab, n, m, max_pivots, as_stream(stream)),
                 "init_state launch");
}

// ---- K1 + K2 ------------------------------------------------------------------
static int validate_split(const char *who, const void *A, const void *b, int n, int m, int64_t ld) {
    SPX_REQUIRE(A && b, "%s: null tableau pointer", who);
    SPX_REQUIRE(n >= 1 && m >= 0, "%s: bad shape n=%d m=%d", who, n, m);
    SPX_REQUIRE(ld >= m && ld >= 16 && ld % 16 == 0, "%s: ld=%lld must be a multiple of 16 >= m", who, (long long)ld);
    SPX_REQUIRE(((uintptr_t)A & 127) == 0, "%s: tableau body must be 128-byte aligned", who);
    return 0;
}

int spx_pick(const double *d_A, const double *d_b, int32_t n, int32_t m, int64_t ld, int32_t rule,
             int32_t sticky, spx_state *d_state, double *d_colbuf, void *stream) {
    if (validate_split("spx_pick", d_A, d_b, n, m, ld)) return -2;
    SPX_REQUIRE(d_state && d_colbuf, "spx_pick: null state/colbuf");
    SPX_REQUIRE(rule == SPX_RULE_REFERENCE || rule == SPX_RULE_DANTZIG, "spx_pick: unknown rule %d", rule);
    return check(spx_launch::pick(d_A, d_b, n, m, ld, rule, sticky, d_state, d_colbuf, as_stream(stream)),
                 "pick launch");
}

// ---- K3 -----------------------------------------------------------------------
int spx_shard_update(const double *d_Ain, double *d_Aout, const double *d_bin, double *d_bout,
                     int32_t n, int32_t m_loc, int64_t ld_loc, int64_t col0, spx_state *d_state,
                     const double *d_colbuf, int32_t *d_rowlab, int32_t *d_collab, int32_t *d_trace,
                     int32_t ahead, void *stream) {
    if (validate_split("spx_update", d_Ain, d_bin, n, m_loc, ld_loc)) return -2;
    if (validate_split("spx_update", d_Aout, d_bout, n, m_loc, ld_loc)) return -2;
    SPX_REQUIRE(d_Ain != d_Aout && d_bin != d_bout, "spx_update: the pivot is out of place; in == out");
    SPX_REQUIRE(d_state && d_colbuf && d_rowlab && d_collab, "spx_update: null state/colbuf/labels");
    SPX_REQUIRE(((uintptr_t)d_colbuf & 15) == 0, "spx_update: colbuf must be 16-byte aligned");
    return check(spx_launch::update(d_Ain, d_Aout, d_bin, d_bout, n, m_loc, ld_loc, col0, d_state, d_colbuf,
                                    d_rowlab, d_collab, d_trace, ahead ? 1 : 0, as_stream(stream)),
                 "update launch");
}

int spx_update(const double *d_Ain, double *d_Aout, const double *d_bin, double *d_bout, int32_t n,
               int32_t m, int64_t ld, spx_state *d_state, const double *d_colbuf, int32_t *d_rowlab,
               int32_t *d_collab, int32_t *d_trace, void *stream) {
    return spx_shard_update(d_Ain, d_Aout, d_bin, d_bout, n, m, ld, 0, d_state, d_colbuf, d_rowlab,
                            d_collab, d_trace, 0, stream);
}

// ---- the pivot loop -------------------------------------------------------------
namespace {

// look-ahead workspace: [second state | second colbuf | candidate message]
struct Workspace {
    spx_state *state2;
    double    *colbuf2;
    double    *msg;
};
inline int64_t align128(int64_t v) { return (v + 127) / 128 * 128; }
int64_t workspace_bytes(int n) {
    return align128(sizeof(spx_state)) + align128(spx_launch::colbuf_doubles(n) * 8) +
           align128(spx_launch::shard_msg_doubles(n) * 8);
}
Workspace carve(void *base, int n) {
    char *p = static_cast<char *>(base);
    Workspace w;
    w.state2 = reinterpret_cast<spx_state *>(p);  p += align128(sizeof(spx_state));
    w.colbuf2 = reinterpret_cast<double *>(p);    p += align128(spx_launch::colbuf_doubles(n) * 8);
    w.msg = reinterpret_cast<double *>(p);
    return w;
}

// one high-priority side stream + fork/join events per device, created on first use
struct SideCtx { cudaStream_t side = nullptr; cudaEvent_t fork = nullptr, join = nullptr; };
SideCtx g_side[64];

int side_ctx(SideCtx **out) {
    int dev = 0;
    if (check(cudaGetDevice(&dev), "cudaGetDevice")) return -1;
    if (dev < 0 || dev >= 64) { set_error("device index %d out of range", dev); return -1; }
    SideCtx &c = g_side[dev];
    if (!c.side) {
        int lo = 0, hi = 0;
        if (check(cudaDeviceGetStreamPriorityRange(&lo, &hi), "priority range")) return -1;
        if (check(cudaStreamCreateWithPriority(&c.side, cudaStreamNonBlocking, hi), "side stream")) return -1;
        if (check(cudaEventCreateWithFlags(&c.fork, cudaEventDisableTiming), "event")) return -1;
        if (check(cudaEventCreateWithFlags(&c.join, cudaEventDisableTiming), "event")) return -1;
    }
    *out = &c;
    return 0;
}

} // namespace

int64_t spx_solve_workspace_bytes(int32_t n) { return workspace_bytes(n); }

int64_t spx_fused_workspace_bytes(int32_t n, int32_t m) {
    return spx_launch::fused_workspace_bytes(n, spx_ld(m));
}

int spx_solve(double *d_A0, double *d_A1, double *d_b0, double *d_b1, int32_t n, int32_t m, int64_t ld,
              int32_t rule, spx_state *d_state, double *d_colbuf, int32_t *d_rowlab, int32_t *d_collab,
              int32_t *d_trace, int32_t chunk, int64_t stop_after, int32_t mode, void *d_work,
              int64_t work_bytes, int32_t *h_status, int64_t *h_npiv, void *stream) {
    if (validate_split("spx_solve", d_A0, d_b0, n, m, ld)) return -2;
    if (validate_split("spx_solve", d_A1, d_b1, n, m, ld)) return -2;
    SPX_REQUIRE(d_state && d_colbuf && d_rowlab && d_collab, "spx_solve: null state/colbuf/labels");
    SPX_REQUIRE(chunk >= 1, "spx_solve: chunk must be >= 1");
    SPX_REQUIRE(rule == SPX_RULE_REFERENCE || rule == SPX_RULE_DANTZIG, "spx_solve: unknown rule %d", rule);
    SPX_REQUIRE(mode >= SPX_LOOP_AUTO && mode <= SPX_LOOP_FUSED, "spx_solve: unknown mode %d", mode);
    if (mode == SPX_LOOP_AUTO) {
        // L2-resident tableaus: one persistent kernel; big ones: look-ahead streaming; else classic
        if (spx_launch::resident_fits(n, m, ld)) mode = SPX_LOOP_RESIDENT;
        else if (d_work != nullptr && ((uintptr_t)d_work & 127) == 0 &&
                 work_bytes >= spx_launch::fused_workspace_bytes(n, ld) &&
                 (int64_t)(n + 1) * ld * 8 >= (256LL << 20)) mode = SPX_LOOP_FUSED;
        // in between (measured, tools/cfg2_lab.py 2000 4000: classic 32, fused 28, look-ahead 23 us/pivot)
        else if (d_work != nullptr && ((uintptr_t)d_work & 127) == 0 && work_bytes >= workspace_bytes(n))
            mode = SPX_LOOP_LOOKAHEAD;
        else mode = SPX_LOOP_CLASSIC;
    }
    SPX_REQUIRE(mode != SPX_LOOP_RESIDENT || spx_launch::resident_fits(n, m, ld),
                "spx_solve: the tableau does not fit the L2-resident loop (n <= 4095, 2 bodies <= 96 MB, cooperative launch)");
    SPX_REQUIRE(mode != SPX_LOOP_LOOKAHEAD || d_work != nullptr, "spx_solve: look-ahead needs a workspace");
    SPX_REQUIRE(mode != SPX_LOOP_FUSED || (d_work != nullptr && ((uintptr_t)d_work & 127) == 0 &&
                                           work_bytes >= spx_launch::fused_workspace_bytes(n, ld)),
                "spx_solve: the fused loop needs a 128-byte aligned workspace of spx_fused_workspace_bytes(n, m) = %lld bytes",
                (long long)spx_launch::fused_workspace_bytes(n, ld));
    const bool ahead = (mode == SPX_LOOP_LOOKAHEAD);
    SPX_REQUIRE(!ahead || (work_bytes >= workspace_bytes(n) && ((uintptr_t)d_work & 127) == 0),
                "spx_solve: workspace must be 128-byte aligned and >= spx_solve_workspace_bytes(n) = %lld bytes",
                (long long)workspace_bytes(n));
    cudaStream_t s = as_stream(stream);
    double *A[2] = {d_A0, d_A1};
    double *b[2] = {d_b0, d_b1};
    spx_state hs;
    if (check(cudaMemcpyAsync(&hs, d_state, sizeof(hs), cudaMemcpyDeviceToHost, s), "read state")) return -1;
    if (check(cudaStreamSynchronize(s), "sync")) return -1;
    if (hs.status == SPX_CAP && hs.npiv < hs.max_pivots) {   // the caller raised the cap: resume
        const int32_t run = SPX_PIVOT;
        if (check(cudaMemcpyAsync(&d_state->status, &run, sizeof(run), cudaMemcpyHostToDevice, s), "resume")) return -1;
        hs.status = SPX_PIVOT;
    }
    SideCtx *sc = nullptr;
    Workspace w{};
    if (ahead) {
        if (side_ctx(&sc)) return -1;
        w = carve(d_work, n);
    }
    int64_t done = 0;
    // the fused passes flip the ping-pong buffers once per PASS, not per pivot: the index of the
    // current buffer travels in the device state while this call runs
    if (mode == SPX_LOOP_FUSED) hs.reserved[0] = hs.npiv & 1;
    bool priced = false;      // look-ahead: d_state/d_colbuf already hold the pick of the current table
    while (hs.status == SPX_PIVOT) {
        int64_t k = chunk;
        if (stop_after > 0 && stop_after - done < k) k = stop_after - done;
        if (k <= 0) break;
        const int64_t base = hs.npiv;
        if (mode == SPX_LOOP_FUSED) {
            // passes of F pivots: price F levels from the stored table, then ONE stream over the body applies
            // them all — 16 B of HBM traffic per cell per F pivots
            const int F = (int)spx_launch::get_option(SPX_OPT_FUSE_DEPTH);
            const int64_t cur = hs.reserved[0] & 1;
            // look-ahead (option): the pricing of pass q+1 runs on a side stream during the update of pass q.
            // Off by default on ONE GPU: pricing is 4 % of a pass there and the overlap costs as much as it
            // hides (measured 3.14 k vs 3.21 k pivots/s); on by default in the column-sharded loop.
            const int la = (int)spx_launch::get_option(SPX_OPT_FUSE_LOOKAHEAD);      // 1 per-pass kernels, 2 persistent engine
            // Without look-ahead, a chunk whose pass count and pivot count differ in parity runs its first pass IN
            // PLACE, so that it leaves table k in buffer k & 1 without a copy of the body.  Only a pass deeper than
            // 8 runs in place: its update kernel reads its own cells coherently (ld_own).  Nothing else reads the
            // body during a pass of this loop.
            const int64_t npass = (k + F - 1) / F;
            const bool inplace = la != 1 && la != 2 && ((cur ^ npass ^ (base + k)) & 1) && (k < F ? k : F) > 8;
            const int64_t reserved = cur | (inplace ? 2 : 0);
            if (check(cudaMemcpyAsync(&d_state->reserved[0], &reserved, sizeof(reserved), cudaMemcpyHostToDevice, s), "cur")) return -1;
            if (la == 1 || la == 2) {
                if (check(spx_launch::fused_solve_passes(d_A0, d_A1, d_b0, d_b1, n, m, ld, rule, d_state, d_work, d_rowlab,
                                                         d_collab, d_trace, k, F,
                                                         (int)spx_launch::get_option(SPX_OPT_FUSE_MIN_BLOCKS), la, s),
                          "fused pass launch")) return -1;
            } else {
                int64_t left = k;
                for (int64_t q = 0; left > 0; ++q) {
                    const int Fp = (int)(left < F ? left : F);
                    const bool same = inplace && q == 0;                 // both tables of the pass are buffer `cur`
                    if (check(spx_launch::fused_pass(same ? A[cur] : d_A0, same ? A[cur] : d_A1, same ? b[cur] : d_b0,
                                                     same ? b[cur] : d_b1, n, m, ld, rule, Fp,
                                                     (int)spx_launch::get_option(SPX_OPT_FUSE_MIN_BLOCKS),
                                                     (int)spx_launch::get_option(SPX_OPT_FUSE_PRICING), 0, d_state, d_work,
                                                     d_rowlab, d_collab, d_trace, s), "fused pass launch")) return -1;
                    left -= Fp;
                }
            }
            if (check(cudaMemcpyAsync(&hs, d_state, sizeof(hs), cudaMemcpyDeviceToHost, s), "read state")) return -1;
            if (check(cudaStreamSynchronize(s), "fused passes")) return -1;
            if (check(spx_launch::fused_solo_sync(), "fused side stream")) return -1;
            done += hs.npiv - base;
            continue;
        }
        if (mode == SPX_LOOP_RESIDENT) {
            // one persistent cooperative launch applies up to k pivots (or all of them)
            if (stop_after <= 0) k = 1LL << 40;
            else k = stop_after - done;
            if (check(spx_launch::resident_loop(d_A0, d_A1, d_b0, d_b1, n, m, ld, rule, k, d_state, d_colbuf,
                                                d_rowlab, d_collab, d_trace, s), "resident launch")) return -1;
            if (check(cudaMemcpyAsync(&hs, d_state, sizeof(hs), cudaMemcpyDeviceToHost, s), "read state")) return -1;
            if (check(cudaStreamSynchronize(s), "resident loop")) return -1;
            done += hs.npiv - base;
            if (hs.status == SPX_PIVOT && hs.npiv == base) break;     // defensive: no progress
            continue;
        }
        if (!ahead) {
            // classic: pick k, update k, pick k+1, ... on one stream
            for (int64_t q = 0; q < k; ++q) {
                const int cur = (int)((base + q) & 1);
                if (check(spx_launch::pick(A[cur], b[cur], n, m, ld, rule, 1, d_state, d_colbuf, s), "pick launch")) return -1;
                if (check(spx_launch::update(A[cur], A[cur ^ 1], b[cur], b[cur ^ 1], n, m, ld, 0, d_state, d_colbuf,
                                             d_rowlab, d_collab, d_trace, 0, s), "update launch")) return -1;
            }
        } else {
            // look-ahead: while update q streams on `s`, the side stream prices pivot q+1 from the
            // same (old) table into the other state/colbuf; the two join before update q+1
            spx_state *S[2] = {d_state, w.state2};
            double *C[2] = {d_colbuf, w.colbuf2};
            if (!priced)
                if (check(spx_launch::pick(A[base & 1], b[base & 1], n, m, ld, rule, 1, d_state, d_colbuf, s), "pick launch")) return -1;
            for (int64_t q = 0; q < k; ++q) {
                const int cur = (int)((base + q) & 1), si = (int)(q & 1);
                if (check(cudaEventRecord(sc->fork, s), "fork")) return -1;
                if (check(cudaStreamWaitEvent(sc->side, sc->fork, 0), "fork wait")) return -1;
                if (check(spx_launch::ahead_candidate(A[cur], b[cur], b[cur ^ 1], n, m, ld, 0, rule, S[si], C[si],
                                                      w.msg, sc->side), "candidate launch")) return -1;
                if (check(spx_launch::ahead_select(w.msg, 1, b[cur ^ 1], n, S[si], S[si ^ 1], C[si ^ 1], nullptr, 0,
                                                   sc->side), "select launch")) return -1;
                if (check(cudaEventRecord(sc->join, sc->side), "join")) return -1;
                if (check(spx_launch::update(A[cur], A[cur ^ 1], b[cur], b[cur ^ 1], n, m, ld, 0, S[si], C[si],
                                             d_rowlab, d_collab, d_trace, 1, s), "update launch")) return -1;
                if (check(cudaStreamWaitEvent(s, sc->join, 0), "join wait")) return -1;
            }
            if (k & 1) {   // the newest state/column sit in the workspace: bring them home
                if (check(cudaMemcpyAsync(d_state, w.state2, sizeof(spx_state), cudaMemcpyDeviceToDevice, s), "state copy")) return -1;
                if (check(cudaMemcpyAsync(d_colbuf, w.colbuf2, (size_t)(n + 1) * sizeof(double),
                                          cudaMemcpyDeviceToDevice, s), "colbuf copy")) return -1;
            }
            priced = true;
        }
        if (check(cudaMemcpyAsync(&hs, d_state, sizeof(hs), cudaMemcpyDeviceToHost, s), "read state")) return -1;
        if (check(cudaStreamSynchronize(s), "pivot chunk")) return -1;
        done += k;
    }
    if (mode == SPX_LOOP_FUSED) {
        // restore the library-wide invariant "the current table is in buffer npiv & 1" (after an in-place first
        // pass, only a call that stopped early or passes of at most 8 levels still need the copy)
        const int cur = (int)(hs.reserved[0] & 1), want = (int)(hs.npiv & 1);
        if (cur != want) {
            if (check(cudaMemcpyAsync(A[want], A[cur], (size_t)(n + 1) * ld * sizeof(double), cudaMemcpyDeviceToDevice, s), "table copy")) return -1;
            if (check(cudaMemcpyAsync(b[want], b[cur], (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, s), "b copy")) return -1;
        }
        const int64_t zero = 0;
        if (check(cudaMemcpyAsync(&d_state->reserved[0], &zero, sizeof(zero), cudaMemcpyHostToDevice, s), "cur")) return -1;
        if (check(cudaStreamSynchronize(s), "sync")) return -1;
    }
    if (h_status) *h_status = hs.status;
    if (h_npiv) *h_npiv = hs.npiv;
    return 0;
}

// one fused pass, or one of its two kernels (bench.py times them separately)
int spx_fused_pass(double *d_A0, double *d_A1, double *d_b0, double *d_b1, int32_t n, int32_t m, int64_t ld,
                   int32_t rule, int32_t depth, int32_t phase, spx_state *d_state, void *d_work, int64_t work_bytes,
                   int32_t *d_rowlab, int32_t *d_collab, int32_t *d_trace, void *stream) {
    if (validate_split("spx_fused_pass", d_A0, d_b0, n, m, ld)) return -2;
    if (validate_split("spx_fused_pass", d_A1, d_b1, n, m, ld)) return -2;
    SPX_REQUIRE(d_state && d_work && d_rowlab && d_collab && ((uintptr_t)d_work & 127) == 0 &&
                work_bytes >= spx_launch::fused_workspace_bytes(n, ld) && depth >= 1 && depth <= spx_launch::fuse_max() &&
                phase >= 0 && phase <= 2, "spx_fused_pass: bad arguments");
    return check(spx_launch::fused_pass(d_A0, d_A1, d_b0, d_b1, n, m, ld, rule, depth,
                                        (int)spx_launch::get_option(SPX_OPT_FUSE_MIN_BLOCKS),
                                        (int)spx_launch::get_option(SPX_OPT_FUSE_PRICING), phase, d_state, d_work,
                                        d_rowlab, d_collab, d_trace, as_stream(stream)), "fused pass launch");
}

// ---- find_optimum / f -----------------------------------------------------------
int spx_extract(const double *d_b, int32_t n, int32_t m, const int32_t *d_collab,
                const double *d_function, double *d_x, double *d_obj, void *stream) {
    SPX_REQUIRE(d_b && d_collab && d_function && d_x && d_obj, "spx_extract: null pointer");
    SPX_REQUIRE(n >= 1 && m >= 1, "spx_extract: bad shape");
    return check(spx_launch::extract(d_b, n, m, d_collab, d_function, d_x, d_obj, as_stream(stream)),
                 "extract launch");
}

// ---- routing of the batched engines (route_lp) ---------------------------------------
int32_t spx_batched_route(int32_t n, int32_t m, int32_t engine) {
    if (!known_engine(engine)) {
        set_error("unknown engine %d", engine);
        return -1;
    }
    if (n < 1 || m < 1) {
        set_error("bad shape %d x %d", n, m);
        return -1;
    }
    Route r;
    if (!route_lp(n, m, engine, 0, &r)) return -1;
    return r.kernel == spx::RAGGED_GLOBAL ? SPX_ENGINE_GLOBAL
                                          : (r.kernel == spx::RAGGED_CLUSTER ? SPX_ENGINE_CLUSTER : SPX_ENGINE_SMEM);
}

// ---- K4 -------------------------------------------------------------------------
int64_t spx_batched_max_cells(void) { return spx_launch::batched_max_cells(); }
int32_t spx_batched_fits(int32_t n, int32_t m) { return spx_launch::batched_fits(n, m) ? 1 : 0; }

int spx_solve_batched(double *d_T, int64_t B, int32_t n, int32_t m, int32_t rule, int32_t max_pivots,
                      double *d_x, double *d_obj, int32_t *d_status, int32_t *d_npiv, int32_t *d_rowlab,
                      int32_t *d_collab, int32_t *d_trace, double *d_snap, void *stream) {
    return solve_uniform("spx_solve_batched", SPX_ENGINE_SMEM, B, n, m, max_pivots,
                         {d_T, nullptr, d_x, d_obj, d_status, d_npiv, d_rowlab, d_collab, d_trace, d_snap, rule, false},
                         stream);
}

// ---- K7 -------------------------------------------------------------------------
int32_t spx_cluster_size(int32_t n, int32_t m) { return spx_launch::cluster_size(n, m); }

int spx_solve_batched_cluster(double *d_T, int64_t B, int32_t n, int32_t m, int32_t rule, int32_t max_pivots,
                              double *d_x, double *d_obj, int32_t *d_status, int32_t *d_npiv, int32_t *d_rowlab,
                              int32_t *d_collab, int32_t *d_trace, double *d_snap, void *stream) {
    return solve_uniform("spx_solve_batched_cluster", SPX_ENGINE_CLUSTER, B, n, m, max_pivots,
                         {d_T, nullptr, d_x, d_obj, d_status, d_npiv, d_rowlab, d_collab, d_trace, d_snap, rule, false},
                         stream);
}

// ---- K8 -------------------------------------------------------------------------
int32_t spx_global_min_cluster_size(int32_t n, int32_t m) { return spx_launch::global_min_cluster_size(n, m); }

int32_t spx_global_cluster_size(int32_t n, int32_t m, int64_t B) {
    int S = 0;
    if (check(spx_launch::global_cluster_size(n, m, B < 0 ? 0 : B, &S), "spx_global_cluster_size")) return -1;
    return S;
}

int spx_solve_batched_global(double *d_T, int64_t B, int32_t n, int32_t m, int32_t rule, int32_t max_pivots,
                             double *d_x, double *d_obj, int32_t *d_status, int32_t *d_npiv, int32_t *d_rowlab,
                             int32_t *d_collab, int32_t *d_trace, double *d_snap, void *stream) {
    return solve_uniform("spx_solve_batched_global", SPX_ENGINE_GLOBAL, B, n, m, max_pivots,
                         {d_T, nullptr, d_x, d_obj, d_status, d_npiv, d_rowlab, d_collab, d_trace, d_snap, rule, false},
                         stream);
}

// ---- ragged batches (K4 + K7 + K8) ---------------------------------------------------
static int64_t ragged_lp_offset() { return ((int64_t)sizeof(spx::RaggedPlan) + 15) / 16 * 16; }

int64_t spx_ragged_plan_bytes(int64_t B) {
    if (B < 0 || B > INT32_MAX) return -1;
    return ragged_lp_offset() + B * (int64_t)sizeof(spx::RaggedLp) + (B * 4 + 15) / 16 * 16;
}

int spx_ragged_plan(const int32_t *h_shapes, int64_t B, int32_t engine, void *h_plan, int64_t plan_bytes,
                    int64_t *h_totals) {
    using namespace spx;
    SPX_REQUIRE(B >= 0 && B <= INT32_MAX, "spx_ragged_plan: bad batch size B = %lld", (long long)B);
    SPX_REQUIRE(known_engine(engine), "spx_ragged_plan: unknown engine %d", engine);
    SPX_REQUIRE(h_plan && h_totals && (B == 0 || h_shapes), "spx_ragged_plan: null shapes/plan/totals");
    SPX_REQUIRE(plan_bytes >= spx_ragged_plan_bytes(B), "spx_ragged_plan: plan_bytes = %lld < spx_ragged_plan_bytes(%lld) = %lld",
                (long long)plan_bytes, (long long)B, (long long)spx_ragged_plan_bytes(B));
    RaggedPlan *P = static_cast<RaggedPlan *>(h_plan);
    RaggedLp *lps = reinterpret_cast<RaggedLp *>(static_cast<char *>(h_plan) + ragged_lp_offset());
    int32_t *order = reinterpret_cast<int32_t *>(lps + B);
    // class of every LP: 0 warp mode, 1 CTA mode, 2 + log2(S) K7, 7 + log2(S) K8; and its shared-memory footprint
    const int forced = forced_cluster_size();
    std::vector<int8_t> cls((size_t)B);
    std::vector<int64_t> bytes((size_t)B);
    int64_t tot[5] = {0, 0, 0, 0, 0};
    for (int64_t k = 0; k < B; ++k) {
        const int32_t n = h_shapes[3 * k], m = h_shapes[3 * k + 1], cap = h_shapes[3 * k + 2];
        SPX_REQUIRE(n >= 1 && m >= 1 && cap >= 0, "spx_ragged_plan: LP %lld: bad shape n=%d m=%d max_pivots=%d",
                    (long long)k, n, m, cap);
        Route r;
        if (!route_lp(n, m, engine, forced, &r)) {
            prefix_error("spx_ragged_plan: LP %lld: ", (long long)k);
            return -2;
        }
        bytes[k] = r.bytes;
        cls[k] = (int8_t)(r.kernel == RAGGED_CLUSTER ? 2 + __builtin_ctz((unsigned)r.S)
                          : r.kernel == RAGGED_GLOBAL ? 7 + __builtin_ctz((unsigned)r.S) : r.kernel);
        const int64_t cells = spx_cells(n, m);
        lps[k] = RaggedLp{n, m, cap, (int32_t)cells, tot[0], tot[1], tot[2], tot[3], tot[4]};
        tot[0] += cells;
        tot[1] += m;
        tot[2] += n;
        tot[3] += cap;
        tot[4] += ((int64_t)cap + 1) * cells;
    }
    // launches: warp mode, CTA mode, K7 by cluster size, then K8 by S_min (or the forced S); inside each, by cells
    // descending, ties by index
    std::vector<int32_t> idx((size_t)B);
    for (int64_t k = 0; k < B; ++k) idx[k] = (int32_t)k;
    std::stable_sort(idx.begin(), idx.end(), [&](int32_t u, int32_t v) {
        return cls[u] != cls[v] ? cls[u] < cls[v] : lps[u].cells > lps[v].cells;
    });
    std::memset(P, 0, sizeof(RaggedPlan));
    int nl = 0;
    for (int64_t q = 0; q < B;) {
        const int c = cls[idx[q]];
        int64_t e = q, big = 0;
        while (e < B && cls[idx[e]] == c) { big = std::max(big, bytes[idx[e]]); ++e; }
        RaggedLaunch &l = P->launch[nl++];
        l.first = q;
        l.count = e - q;
        l.S = 1;
        l.per_cta = 1;
        if (c == RAGGED_WARP) {
            const int64_t slot = (big + 15) / 16 * 16;
            l.kernel = RAGGED_WARP;
            l.per_cta = spx_launch::ragged_warps_per_cta(slot, l.count);
            l.threads = 32 * l.per_cta;
            l.smem = slot * l.per_cta;
            l.slot_doubles = slot / 8;
        } else if (c == RAGGED_CTA) {
            l.kernel = RAGGED_CTA;
            l.threads = spx_launch::ragged_cta_threads(lps[idx[q]].cells);     // the largest LP comes first
            l.smem = big;
        } else {
            l.kernel = c < 7 ? RAGGED_CLUSTER : RAGGED_GLOBAL;
            l.S = 1 << (c < 7 ? c - 2 : c - 7);
            l.threads = 512;
            l.smem = big;
            l.pick_S = (l.kernel == RAGGED_GLOBAL && forced == 0) ? 1 : 0;
            SPX_REQUIRE(l.count <= INT32_MAX / l.S, "spx_ragged_plan: %lld LPs x S = %d CTAs exceed one grid",
                        (long long)l.count, l.S);
        }
        q = e;
    }
    std::copy(idx.begin(), idx.end(), order);
    P->magic = RAGGED_MAGIC;
    P->abi = SPX_ABI_VERSION;
    P->B = B;
    P->engine = engine;
    P->nlaunch = nl;
    for (int i = 0; i < 5; ++i) P->totals[i] = h_totals[i] = tot[i];
    P->lp_offset = ragged_lp_offset();
    P->order_offset = ragged_lp_offset() + B * (int64_t)sizeof(RaggedLp);
    return 0;
}

// the launch list of a plan covers its B LPs exactly once, in order
static bool ragged_header_sane(const spx::RaggedPlan *P) {
    using namespace spx;
    int64_t counted = 0;
    bool sane = P->B >= 0 && P->nlaunch >= 0 && P->nlaunch <= RAGGED_MAX_LAUNCHES &&
                P->lp_offset == ragged_lp_offset() && P->order_offset == P->lp_offset + P->B * (int64_t)sizeof(RaggedLp);
    for (int i = 0; sane && i < P->nlaunch; ++i) {
        const RaggedLaunch &l = P->launch[i];
        sane = l.first == counted && l.count >= 1 && l.kernel >= RAGGED_WARP && l.kernel <= RAGGED_GLOBAL &&
               l.per_cta >= 1 && l.threads >= 32 && l.S >= 1 && l.S <= 16 && (l.pick_S == 0 || l.kernel == RAGGED_GLOBAL);
        counted += l.count;
    }
    return sane && counted == P->B;
}

// The plan `who` was given, checked (magic, ABI version and launch list), as a view of its host copy h_plan and of its
// device copy d_plan (null: the view's device arrays are null); false, with the error set, when it is not a plan
static bool checked_plan(const char *who, const void *h_plan, const void *d_plan, spx::PlanView *v) {
    using namespace spx;
    if (!h_plan) {
        set_error("%s: null plan", who);
        return false;
    }
    const RaggedPlan *P = static_cast<const RaggedPlan *>(h_plan);
    if (P->magic != RAGGED_MAGIC || P->abi != SPX_ABI_VERSION) {
        set_error("%s: h_plan is not a plan of this library (magic / ABI version mismatch)", who);
        return false;
    }
    if (!ragged_header_sane(P)) {
        set_error("%s: inconsistent plan header (B = %lld)", who, (long long)P->B);
        return false;
    }
    auto at = [](const void *plan, int64_t offset) {
        return plan ? static_cast<const char *>(plan) + offset : nullptr;
    };
    *v = PlanView{P, reinterpret_cast<const RaggedLp *>(at(h_plan, P->lp_offset)),
                  reinterpret_cast<const int32_t *>(at(h_plan, P->order_offset)),
                  reinterpret_cast<const RaggedLp *>(at(d_plan, P->lp_offset)),
                  reinterpret_cast<const int32_t *>(at(d_plan, P->order_offset))};
    return true;
}

// One ragged solve (io.warm == false) or resume (io.warm == true): the body of spx_solve_batched_ragged and
// spx_warm_solve_ragged
static int solve_ragged(const char *who, const void *h_plan, const void *d_plan, const spx::BatchIO &io,
                        void *stream) {
    using namespace spx;
    PlanView v;
    if (!checked_plan(who, h_plan, d_plan, &v)) return -2;
    if (v.P->B == 0) return 0;
    SPX_REQUIRE(d_plan && io.T && io.status && io.npiv, "%s: null d_plan/T/status/npiv", who);
    SPX_REQUIRE(!io.warm || (io.rowlab && io.collab), "%s: null rowlab/collab (the labels to resume from)", who);
    SPX_REQUIRE(!io.warm || !io.obj || io.function, "%s: null function with obj", who);
    SPX_REQUIRE(io.rule == SPX_RULE_REFERENCE || io.rule == SPX_RULE_DANTZIG, "%s: unknown rule %d", who, io.rule);
    cudaStream_t s = as_stream(stream);
    char what[96];
    for (int i = 0; i < v.P->nlaunch; ++i) {
        const RaggedLaunch &l = v.P->launch[i];
        if (l.kernel == RAGGED_GLOBAL) {
            int S = 0;
            int64_t smem = 0;
            snprintf(what, sizeof(what), "%s: occupancy", who);
            if (check(spx_launch::ragged_global_size(v, l, &S, &smem), what))
                return -1;
            SPX_REQUIRE(l.count <= INT32_MAX / S, "%s: %lld LPs x S = %d CTAs exceed one grid", who,
                        (long long)l.count, S);
            if (check_cluster_launch(spx_launch::solve_ragged_global(v, l, S, smem, io, s), who, S, smem))
                return -1;
        } else if (l.kernel == RAGGED_CLUSTER) {
            if (check_cluster_launch(spx_launch::solve_ragged_cluster(v, l, io, s), who, l.S, l.smem))
                return -1;
        } else if (check(spx_launch::solve_ragged_batched(v, l, io, s), "ragged batched launch")) {
            return -1;
        }
    }
    return 0;
}

int spx_solve_batched_ragged(double *d_T, const void *h_plan, const void *d_plan, int32_t rule, double *d_x,
                             double *d_obj, int32_t *d_status, int32_t *d_npiv, int32_t *d_rowlab, int32_t *d_collab,
                             int32_t *d_trace, double *d_snap, void *stream) {
    return solve_ragged("spx_solve_batched_ragged", h_plan, d_plan,
                        {d_T, nullptr, d_x, d_obj, d_status, d_npiv, d_rowlab, d_collab, d_trace, d_snap, rule, false},
                        stream);
}

int32_t spx_ragged_cluster_size(const void *h_plan, int32_t launch) {
    spx::PlanView v;
    if (!checked_plan("spx_ragged_cluster_size", h_plan, nullptr, &v)) return -1;
    if (launch < 0 || launch >= v.P->nlaunch) {
        set_error("spx_ragged_cluster_size: launch %d of a plan of %d launches", launch, v.P->nlaunch);
        return -1;
    }
    const spx::RaggedLaunch &l = v.P->launch[launch];
    if (l.kernel != spx::RAGGED_GLOBAL) return l.S;
    int S = 0;
    int64_t smem = 0;
    if (check(spx_launch::ragged_global_size(v, l, &S, &smem), "spx_ragged_cluster_size")) return -1;
    return S;
}

// ---- sensitivity report of optimal final tables (csrc/spx_sensitivity.cu) -------------
int spx_sensitivity_batched(const double *d_T, int64_t B, int32_t n, int32_t m, const int32_t *d_status,
                            const int32_t *d_rowlab, const int32_t *d_collab, double *d_dual, double *d_slack,
                            double *d_redcost, double *d_rhs_range, double *d_cost_range, void *stream) {
    SPX_REQUIRE(B >= 0 && n >= 1 && m >= 1, "spx_sensitivity_batched: bad arguments (B = %lld, n = %d, m = %d)",
                (long long)B, n, m);
    if (B == 0) return 0;
    SPX_REQUIRE(d_T && d_status && d_rowlab && d_collab, "spx_sensitivity_batched: null T/status/rowlab/collab");
    return check(spx_launch::sensitivity_uniform(d_T, B, n, m, d_status, d_rowlab, d_collab, d_dual, d_slack,
                                                 d_redcost, d_rhs_range, d_cost_range, as_stream(stream)),
                 "sensitivity launch");
}

int spx_sensitivity_ragged(const double *d_T, const void *h_plan, const void *d_plan, const int32_t *d_status,
                           const int32_t *d_rowlab, const int32_t *d_collab, double *d_dual, double *d_slack,
                           double *d_redcost, double *d_rhs_range, double *d_cost_range, void *stream) {
    spx::PlanView v;
    if (!checked_plan("spx_sensitivity_ragged", h_plan, d_plan, &v)) return -2;
    if (v.P->B == 0) return 0;
    SPX_REQUIRE(d_plan && d_T && d_status && d_rowlab && d_collab,
                "spx_sensitivity_ragged: null d_plan/T/status/rowlab/collab");
    return check(spx_launch::sensitivity_ragged(v, d_T, d_status, d_rowlab, d_collab, d_dual, d_slack, d_redcost,
                                                d_rhs_range, d_cost_range, as_stream(stream)),
                 "ragged sensitivity launch");
}

int spx_sensitivity_split(const double *d_A, const double *d_b, int32_t n, int32_t m, int64_t ld,
                          const int32_t *d_rowlab, const int32_t *d_collab, double *d_dual, double *d_slack,
                          double *d_redcost, double *d_rhs_range, double *d_cost_range, int32_t *h_optimal,
                          void *stream) {
    SPX_REQUIRE(n >= 1 && m >= 1 && ld >= m, "spx_sensitivity_split: bad arguments (n = %d, m = %d, ld = %lld)", n, m,
                (long long)ld);
    SPX_REQUIRE(d_A && d_b && d_rowlab && d_collab && h_optimal, "spx_sensitivity_split: null A/b/rowlab/collab/optimal");
    // pick_element's tests, simplex.py:72-76 and :94-98: optimal when no b cell and no f cell is negative
    cudaStream_t s = as_stream(stream);
    std::vector<double> hb((size_t)n), hf((size_t)m);
    if (check(cudaMemcpyAsync(hb.data(), d_b, sizeof(double) * n, cudaMemcpyDeviceToHost, s), "spx_sensitivity_split: copy b") ||
        check(cudaMemcpyAsync(hf.data(), d_A + (int64_t)n * ld, sizeof(double) * m, cudaMemcpyDeviceToHost, s),
              "spx_sensitivity_split: copy f") ||
        check(cudaStreamSynchronize(s), "spx_sensitivity_split: synchronize"))
        return -1;
    int optimal = 1;
    for (double v : hb) optimal &= !(v < 0);
    for (double v : hf) optimal &= !(v < 0);
    *h_optimal = optimal;
    return check(spx_launch::sensitivity_split(d_A, d_b, n, m, ld, optimal, d_rowlab, d_collab, d_dual, d_slack,
                                               d_redcost, d_rhs_range, d_cost_range, s),
                 "split sensitivity launch");
}

// ---- certificates of infeasible and unbounded LPs (csrc/spx_certificate.cu) ----------
// d_farkas and d_ray are the workspace of their halves: the index and bound of a half need its vector
static bool cert_outputs_ok(const char *who, const int32_t *row, const double *farkas, const double *bound,
                            const int32_t *col, const double *ray, const double *slope) {
    if ((row || bound) && !farkas) {
        set_error("%s: d_row and d_bound need d_farkas (the workspace of the Farkas half)", who);
        return false;
    }
    if ((col || slope) && !ray) {
        set_error("%s: d_col and d_slope need d_ray (the workspace of the ray half)", who);
        return false;
    }
    return true;
}

int spx_certificate_batched(const double *d_T, int64_t B, int32_t n, int32_t m, const int32_t *d_rowlab,
                            const int32_t *d_collab, int32_t *d_row, double *d_farkas, double *d_bound,
                            int32_t *d_col, double *d_ray, double *d_slope, void *stream) {
    SPX_REQUIRE(B >= 0 && n >= 1 && m >= 1, "spx_certificate_batched: bad arguments (B = %lld, n = %d, m = %d)",
                (long long)B, n, m);
    if (!cert_outputs_ok("spx_certificate_batched", d_row, d_farkas, d_bound, d_col, d_ray, d_slope)) return -2;
    if (B == 0) return 0;
    SPX_REQUIRE(d_T && d_rowlab && d_collab, "spx_certificate_batched: null T/rowlab/collab");
    return check(spx_launch::certificate_uniform(d_T, B, n, m, d_rowlab, d_collab, d_row, d_farkas, d_bound, d_col,
                                                 d_ray, d_slope, as_stream(stream)),
                 "certificate launch");
}

int spx_certificate_ragged(const double *d_T, const void *h_plan, const void *d_plan, const int32_t *d_rowlab,
                           const int32_t *d_collab, int32_t *d_row, double *d_farkas, double *d_bound,
                           int32_t *d_col, double *d_ray, double *d_slope, void *stream) {
    spx::PlanView v;
    if (!checked_plan("spx_certificate_ragged", h_plan, d_plan, &v)) return -2;
    if (!cert_outputs_ok("spx_certificate_ragged", d_row, d_farkas, d_bound, d_col, d_ray, d_slope)) return -2;
    if (v.P->B == 0) return 0;
    SPX_REQUIRE(d_plan && d_T && d_rowlab && d_collab, "spx_certificate_ragged: null d_plan/T/rowlab/collab");
    return check(spx_launch::certificate_ragged(v, d_T, d_rowlab, d_collab, d_row, d_farkas, d_bound, d_col, d_ray,
                                                d_slope, as_stream(stream)),
                 "ragged certificate launch");
}

int spx_certificate_split(const double *d_A, const double *d_b, int32_t n, int32_t m, int64_t ld,
                          const int32_t *d_rowlab, const int32_t *d_collab, int32_t *d_row, double *d_farkas,
                          double *d_bound, int32_t *d_col, double *d_ray, double *d_slope, void *stream) {
    SPX_REQUIRE(n >= 1 && m >= 1 && ld >= m, "spx_certificate_split: bad arguments (n = %d, m = %d, ld = %lld)", n, m,
                (long long)ld);
    SPX_REQUIRE(d_A && d_b && d_rowlab && d_collab, "spx_certificate_split: null A/b/rowlab/collab");
    if (!cert_outputs_ok("spx_certificate_split", d_row, d_farkas, d_bound, d_col, d_ray, d_slope)) return -2;
    return check(spx_launch::certificate_split(d_A, d_b, n, m, ld, d_rowlab, d_collab, d_row, d_farkas, d_bound, d_col,
                                               d_ray, d_slope, as_stream(stream)),
                 "split certificate launch");
}

// ---- warm start: change and resume final tables (csrc/spx_warm.cu) ------------------
int spx_warm_change_batched(double *d_T, int64_t B, int32_t n, int32_t m, const int32_t *d_rowlab,
                            const int32_t *d_collab, const double *d_delta_b, const double *d_delta_c, void *stream) {
    SPX_REQUIRE(B >= 0 && n >= 1 && m >= 1, "spx_warm_change_batched: bad arguments (B = %lld, n = %d, m = %d)",
                (long long)B, n, m);
    if (B == 0 || (!d_delta_b && !d_delta_c)) return 0;
    SPX_REQUIRE(d_T && d_rowlab && d_collab, "spx_warm_change_batched: null T/rowlab/collab");
    return check(spx_launch::warm_change_uniform(d_T, B, n, m, d_rowlab, d_collab, d_delta_b, d_delta_c,
                                                 as_stream(stream)),
                 "warm change launch");
}

int spx_warm_change_ragged(double *d_T, const void *h_plan, const void *d_plan, const int32_t *d_rowlab,
                           const int32_t *d_collab, const double *d_delta_b, const double *d_delta_c, void *stream) {
    spx::PlanView v;
    if (!checked_plan("spx_warm_change_ragged", h_plan, d_plan, &v)) return -2;
    if (v.P->B == 0 || (!d_delta_b && !d_delta_c)) return 0;
    SPX_REQUIRE(d_plan && d_T && d_rowlab && d_collab, "spx_warm_change_ragged: null d_plan/T/rowlab/collab");
    return check(spx_launch::warm_change_ragged(v, d_T, d_rowlab, d_collab, d_delta_b, d_delta_c, as_stream(stream)),
                 "ragged warm change launch");
}

int spx_warm_solve_batched(int32_t engine, double *d_T, int64_t B, int32_t n, int32_t m, int32_t rule,
                           int32_t max_pivots, const double *d_function, double *d_x, double *d_obj,
                           int32_t *d_status, int32_t *d_npiv, int32_t *d_rowlab, int32_t *d_collab,
                           int32_t *d_trace, double *d_snap, void *stream) {
    return solve_uniform("spx_warm_solve_batched", engine, B, n, m, max_pivots,
                         {d_T, d_function, d_x, d_obj, d_status, d_npiv, d_rowlab, d_collab, d_trace, d_snap, rule, true},
                         stream);
}

int spx_warm_solve_ragged(double *d_T, const void *h_plan, const void *d_plan, int32_t rule,
                          const double *d_function, double *d_x, double *d_obj, int32_t *d_status,
                          int32_t *d_npiv, int32_t *d_rowlab, int32_t *d_collab, int32_t *d_trace,
                          double *d_snap, void *stream) {
    return solve_ragged("spx_warm_solve_ragged", h_plan, d_plan,
                        {d_T, d_function, d_x, d_obj, d_status, d_npiv, d_rowlab, d_collab, d_trace, d_snap, rule, true},
                        stream);
}

// ---- column-sharded flow ----------------------------------------------------------
int64_t spx_shard_msg_doubles(int32_t n) { return spx_launch::shard_msg_doubles(n); }

int spx_shard_candidate(const double *d_A, const double *d_b, int32_t n, int32_t m_loc, int64_t ld_loc,
                        int64_t col0, int32_t rule, int32_t sticky, spx_state *d_state, double *d_send,
                        void *stream) {
    if (validate_split("spx_shard_candidate", d_A, d_b, n, m_loc, ld_loc)) return -2;
    SPX_REQUIRE(d_state && d_send && col0 >= 0, "spx_shard_candidate: bad arguments");
    SPX_REQUIRE(rule == SPX_RULE_REFERENCE || rule == SPX_RULE_DANTZIG, "spx_shard_candidate: unknown rule %d", rule);
    return check(spx_launch::shard_candidate(d_A, d_b, n, m_loc, ld_loc, col0, rule, sticky, d_state, d_send,
                                             as_stream(stream)), "candidate launch");
}

int spx_shard_select(const double *d_gathered, int32_t nranks, const double *d_b, int32_t n, int32_t rule,
                     int32_t sticky, spx_state *d_state, double *d_colbuf, const uint64_t *d_flags,
                     uint64_t seq, void *stream) {
    (void)rule;
    SPX_REQUIRE(d_gathered && d_b && d_state && d_colbuf && nranks >= 1 && n >= 1,
                "spx_shard_select: bad arguments");
    return check(spx_launch::shard_select(d_gathered, nranks, d_b, n, sticky, d_state, d_colbuf,
                                          reinterpret_cast<const unsigned long long *>(d_flags), seq,
                                          as_stream(stream)), "select launch");
}

int spx_ahead_candidate(const double *d_A, const double *d_bin, double *d_bout, int32_t n, int32_t m_loc,
                        int64_t ld_loc, int64_t col0, int32_t rule, const spx_state *d_state,
                        const double *d_colbuf, double *d_send, void *stream) {
    if (validate_split("spx_ahead_candidate", d_A, d_bin, n, m_loc, ld_loc)) return -2;
    SPX_REQUIRE(d_bout && d_bout != d_bin && d_state && d_colbuf && d_send && col0 >= 0,
                "spx_ahead_candidate: bad arguments");
    SPX_REQUIRE(rule == SPX_RULE_REFERENCE || rule == SPX_RULE_DANTZIG, "spx_ahead_candidate: unknown rule %d", rule);
    return check(spx_launch::ahead_candidate(d_A, d_bin, d_bout, n, m_loc, ld_loc, col0, rule, d_state, d_colbuf,
                                             d_send, as_stream(stream)), "candidate launch");
}

int spx_ahead_select(const double *d_gathered, int32_t nranks, const double *d_bnext, int32_t n,
                     const spx_state *d_state_cur, spx_state *d_state_next, double *d_colbuf_next,
                     const uint64_t *d_flags, uint64_t seq, void *stream) {
    SPX_REQUIRE(d_gathered && d_bnext && d_state_cur && d_state_next && d_colbuf_next && nranks >= 1 && n >= 1 &&
                d_state_cur != d_state_next, "spx_ahead_select: bad arguments");
    return check(spx_launch::ahead_select(d_gathered, nranks, d_bnext, n, d_state_cur, d_state_next,
                                          d_colbuf_next, reinterpret_cast<const unsigned long long *>(d_flags),
                                          seq, as_stream(stream)), "select launch");
}

} // extern "C"
