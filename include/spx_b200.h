/*
 * spx_b200.h — C ABI of libspx_b200.so: the B200 (sm_100a) tableau pivot loop.
 *
 * The reference (jqnfxa/Simplex-Method-Solver) is pure Python and has no FFI;
 * its boundary for this path is the Python surface of src/simplex.py.  Each
 * entry point below names the reference code it replaces (file:line into
 * /root/reference/src/).  INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error (text: spx_last_error());
 *   - all pointers named d_* are DEVICE pointers (plain void* / double* taken
 *     from any allocator, e.g. torch.Tensor.data_ptr()); h_* are HOST pointers;
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream);
 *   - nothing allocates behind the caller's back;
 *   - all arithmetic is IEEE binary64 with separately rounded mul/sub/div
 *     (no FMA contraction, no reciprocal multiply) so results are bit-identical
 *     to CPython floats (simplex.py:156,160,163,173-175).
 *
 * Device data layouts
 *   "reference flat"  the reference's ragged table flattened row-major: n rows
 *                     of m+1 cells [a_1..a_m, b] then the f row with m cells
 *                     (simplex.py:36-39); cells = n*(m+1)+m.  Used by the
 *                     batched small-LP solver and by import/export.
 *   "split"           used by the streaming solver for large tableaus:
 *                     body  A[(n+1)][ld]  row-major, columns 0..m-1, row n = f,
 *                           ld = spx_ld(m) (multiple of 16 doubles => every row
 *                           starts on a 128-byte line, m+1 = 32769 would not);
 *                     rhs   b[n] contiguous (the '-b' column), kept separate so
 *                           the body is a clean m-wide stream and, when the
 *                           body is column-sharded over GPUs, b is replicated.
 *   colbuf            the gathered pivot column, spx_colbuf_doubles(n) doubles
 *                     (n+1 cells, f row last, padded to a whole row tile).
 *   labels            int32 codes instead of the reference's strings
 *                     (simplex.py:30-33): x_j -> j-1, y_i -> m+i-1; rowlab[m]
 *                     is the header over the columns, collab[n] labels the rows.
 */
#ifndef SPX_B200_H
#define SPX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPX_ABI_VERSION 8

/* status codes == the outcomes of pick_element(), simplex.py:70-141 */
#define SPX_PIVOT       1   /* (True, r, c, e)                                   :91,:141 */
#define SPX_OPTIMAL     0   /* (False, x1, x2, f)                                :101-103 */
#define SPX_INCORRECT  -1   /* ValueError("incorrect system")                    :88-89   */
#define SPX_NOCONV     -2   /* ValueError("simplex method does not converge")    :138-139 */
#define SPX_CAP        -3   /* max_pivots reached; the reference has no cap and cycles    */
#define SPX_PEER_TIMEOUT -4 /* column-sharded flow: a peer's message did not arrive in 20 s */

/* pivoting rules */
#define SPX_RULE_REFERENCE 0  /* first-negative entering, max-negative-ratio leaving (the reference) */
#define SPX_RULE_DANTZIG   1  /* most-negative entering (lowest index on ties); leaving as reference */
/* Devex reference weights (Forrest-Goldfarb): the candidate f_j < 0 with the largest f_j^2 / w_j enters (NaN scores
 * below every number, lowest j on ties); after every pivot (r, c), phase-1 pivots included, w_j = max(w_j,
 * u_j^2 * w_c) and w_c = max(1, u_c^2 * w_c), u = the new pivot row; every solve and every resume starts from w = 1.
 * Phase 1, the leaving row and the pivot arithmetic are the reference's.  Batched entries only
 * (spx_solve_batched, spx_solve_batched_cluster, spx_solve_batched_global, spx_solve_batched_ragged,
 * spx_warm_solve_batched, spx_warm_solve_ragged): there d_x is required, it is the weights' workspace until the
 * epilogue writes x.  Every single-LP and sharded entry rejects it. */
#define SPX_RULE_DEVEX     2
/* Dantzig with Bland's rule on degenerate pivots, and a ratio-tested phase 1.  t = the lowest row with b < 0.  Phase 1
 * (t exists): the candidates are the j with T[t][j] > 0 (none: SPX_INCORRECT); phase 2: the j with f_j < 0 (none:
 * SPX_OPTIMAL).  c_D = the candidate with the largest T[t][j] (phase 1) or -f_j (phase 2), lowest j on ties; c_B = the
 * candidate with the lowest header label.  The leaving row of column c is the least (ratio, not target, row label, i)
 * over row t (ratio (0 - b_t) / T[t][c]) and the rows i != t with T[i][c] < 0 and !(b_i < 0) (ratio
 * b_i / (0 - T[i][c])); ratios compare by value, -0 = +0, NaN after every number; no row: SPX_NOCONV.  The pivot is
 * (leave(c_D), c_D) unless that ratio is +-0, then (leave(c_B), c_B).  A feasible row stays feasible, and the rule
 * ends in exact arithmetic (DESIGN.md, "Dantzig with Bland's rule on degenerate pivots").  Stateless: a capped solve
 * and its resume pivot as one uncapped solve.  Batched entries only, as SPX_RULE_DEVEX, without its need of d_x. */
#define SPX_RULE_DANTZIG_BLAND 4
/* 3 is not a rule: every entry refuses it as unknown */

/* Device-resident solver state, 128 bytes.  Written by the pick kernels, read
 * by the update kernels, so a whole chunk of pivots can be enqueued with no host
 * round trip; once status != SPX_PIVOT every later kernel of the chunk is a no-op. */
typedef struct spx_state {
    int32_t status;       /* outcome of the most recent pick (SPX_PIVOT while running)  */
    int32_t r;            /* pivot row    (valid when status == SPX_PIVOT)              */
    int64_t c;            /* pivot column (GLOBAL index when column-sharded)            */
    double  p;            /* pivot value T[r][c]                                        */
    int64_t npiv;         /* pivots applied so far                                      */
    int64_t max_pivots;   /* cap; pick reports SPX_CAP when npiv has reached it         */
    int32_t phase1;       /* 1 when the pivot came from the '-b' branch (:79-91)        */
    int32_t slot;         /* hint slot the next update fills = (npiv+1)&1               */
    /* fused pricing: while update k writes the new f row and b column it also
     * min-reduces the first negative index of each into hint_*[slot]; the next
     * pick uses them when hint_tag[npiv&1] == npiv, else it scans.              */
    int64_t hint_tag[2];
    int32_t hint_bneg[2]; /* first i with b[i] < 0, INT32_MAX none                      */
    int32_t hint_fneg[2]; /* first LOCAL j with f[j] < 0, INT32_MAX none                */
    int64_t reserved[6];  /* [0]: fused loops only — index (0/1) of the ping-pong buffer holding table npiv
                           *      (they flip once per PASS, not per pivot); 0 elsewhere                   */
} spx_state;

/* ---- library ----------------------------------------------------------- */
int         spx_version(void);               /* SPX_ABI_VERSION */
const char *spx_last_error(void);            /* thread-local text of the last failure */
int64_t     spx_ld(int64_t m);               /* leading dimension (doubles) of a split body of m columns */
int64_t     spx_cells(int32_t n, int32_t m); /* n*(m+1)+m */
int64_t     spx_colbuf_doubles(int32_t n);   /* capacity a pivot-column buffer needs */
int         spx_state_bytes(void);           /* sizeof(spx_state) */
int         spx_device_info(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor);
/* kernels of this library launched since the last call with reset != 0 (bench.py's gpu_launches) */
int64_t     spx_launch_count(int reset);

/* process-wide tuning knobs; every setting computes bit-identical results */
/* Keys 1, 3, 4, 10 and 15 are retired: they selected kernel variants that measured slower than the defaults and
 * were removed.  spx_set_option rejects them with any value and spx_get_option reads 0; the numbers are never reused. */
#define SPX_OPT_TILED_MIN_BLOCKS 2  /* tiled kernel: resident CTAs per SM the register budget targets (1..4) */
#define SPX_OPT_TILED_ROWS       5  /* tiled kernel rows per tile (0 = auto; else a multiple of 8 <= 64) */
#define SPX_OPT_FUSE_DEPTH       6  /* one-GPU fused loop: pivots per pass over the body: 1-8 or 16 (0 = default 16;
                                         spx_get_option reads the depth in use).  The column-sharded loop and
                                         look-ahead pricing apply at most 8 */
#define SPX_OPT_FUSE_MIN_BLOCKS  7  /* fused update kernel: resident CTAs per SM its register budget targets (2..4, 0 = default 3) */
#define SPX_OPT_FUSE_PRICING     8  /* fused loop pricing kernel: 0 auto, 1 one CTA, 2 whole-GPU cooperative */
#define SPX_OPT_FUSE_LOOKAHEAD   9  /* fused loop in spx_solve: 1 = price pass q+1 on a side stream during update q, 2 = the same with the persistent pricing engine (see spx_fshard_set_lookahead); default 0: off on one GPU */
#define SPX_OPT_FUSE_TILE_ROWS   11 /* fused update kernel: rows of the strip one warp walks (0 = 128; a multiple of 8 <= 4096) */
#define SPX_OPT_SHARD_THREADS    13 /* sharded / look-ahead pricing kernel: threads per CTA, one CTA per SM (0 = default 512; 64..512, multiple of 32) */
#define SPX_OPT_SHARD_CTAS       14 /* sharded / look-ahead pricing kernel: at most this many CTAs (0 = one per SM) */
#define SPX_OPT_FUSE_PAIRS       12 /* fused update kernel: column pairs per lane, i.e. strip width / 64 (0 = default 2; 1 or 2) */
#define SPX_OPT_CLUSTER_SIZE     16 /* K7 and K8 (spx_solve_batched_cluster, spx_solve_batched_global, and ragged plans, read when the plan is made): CTAs per LP, 1, 2, 4, 8 or 16 (0 = default: spx_cluster_size(n, m) for K7, spx_global_cluster_size(n, m, B) for K8, spx_ragged_cluster_size for a ragged K8 launch); a size whose footprint does not fit is rejected */
int         spx_set_option(int32_t option, int64_t value);
int64_t     spx_get_option(int32_t option);
/* Device self-test of the hoisted-reciprocal division used by K3 against the
 * compiler's div.rn.f64: for k < count compares d_a[k] / d_p[k % np]; returns the
 * number of bit mismatches in *h_mismatches (and the first offending pair). */
int         spx_selftest_division(const double *d_a, const double *d_p, int64_t count, int64_t np,
                                  uint64_t *h_mismatches, double *h_first_bad, void *stream);
/* Device self-test of the fused update's LAZY range guard (csrc/spx_fused.cu, update_lazy_kernel): chain k < count
 * takes the cell d_t0[k] through `levels` (1..8) pending pivots — pivot values d_p[levels], pivot-row values
 * d_rj[count][levels], pivot-column values d_ci[count][levels], i.e. `levels` applications of
 * recalculate_matrix()'s cell formula (simplex.py:173-175) — once the kernel's way (unguarded fast divisions, ONE
 * range test on the result, guarded re-do when it fails) into d_out_lazy, once with every division guarded into
 * d_out_ref.  Chains deeper than 8 levels take the depth-16 kernel's way: a range test after each group of 8, and the
 * two-operation quotient on the levels whose divisor it flags (spx_selftest_two_op).  The caller compares the bits.
 * *h_redo = how many chains took the re-do. */
int         spx_selftest_lazy_guard(const double *d_t0, const double *d_p, const double *d_rj, const double *d_ci,
                                    int32_t levels, int64_t count, double *d_out_lazy, double *d_out_ref,
                                    uint64_t *h_redo, void *stream);
/* Device self-test of the one-GPU fused update's two-operation quotient (csrc/spx_fused.cu, two_op_flag): for each
 * divisor d_p[k < np], d_flags[k] = 1 when the update kernel would divide by it with fma(a, yh, RN(a * yl)), else 0.
 * For every flagged divisor the quotient is compared bit for bit with div.rn.f64 on every candidate numerator at
 * K = 64 and on per_p pseudo-random numerators; *h_mismatches = the number of differences (0 expected). */
int         spx_selftest_two_op(const double *d_p, int64_t np, int64_t per_p, int32_t *d_flags,
                                uint64_t *h_mismatches, void *stream);

/* ---- layout conversion (SimplexMethod.__init__, simplex.py:25-39) -------- */
/* src_rows is the reference's `constraints` as a dense row-major [n][m+1] fp64
 * array, src_function its `function` [m]; both host or device
 * (cudaMemcpyDefault).  For a reference-flat buffer pass
 * src_function = src_rows + n*(m+1).  dst is split; the padding columns of d_A
 * are zeroed.  Host sources should be pinned for full PCIe bandwidth. */
int spx_import_table(const double *src_rows, const double *src_function, double *d_A, double *d_b,
                     int32_t n, int32_t m, int64_t ld, void *stream);
/* Column block [col0, col0+m_loc) of the same source -> a local split body
 * d_A[(n+1)][ld_loc] (+ b when d_b != NULL): the loader of one column shard.
 * The source pitch is m + 1 cells and b is its column m; m = 0 (with m_loc = 0)
 * describes the packed block of a rank that owns no columns: b alone, pitch 8 bytes. */
int spx_import_shard(const double *src_rows, const double *src_function, double *d_A, double *d_b,
                     int32_t n, int32_t m, int64_t col0, int32_t m_loc, int64_t ld_loc,
                     void *stream);
/* split -> [n][m+1] rows + [m] f row (host or device destinations): what
 * Info.table / SimplexMethod.table expose (simplex.py:16,36-39). */
int spx_export_table(const double *d_A, const double *d_b, double *dst_rows, double *dst_function,
                     int32_t n, int32_t m, int64_t ld, void *stream);
/* state = {running, npiv 0, cap}, labels x1..xm / y1..yn (simplex.py:30-33) */
int spx_init_state(spx_state *d_state, int32_t *d_rowlab, int32_t *d_collab,
                   int32_t n, int32_t m, int64_t max_pivots, void *stream);

/* ---- K1 + K2: pick_element(), simplex.py:70-141 -------------------------- */
/* Selects the pivot of the split tableau (d_A, d_b); writes *d_state and gathers
 * the pivot column (n+1 doubles, f row last) into d_colbuf for spx_update.
 * sticky != 0: do nothing when d_state->status is already terminal (used by
 * pre-enqueued chunks). */
int spx_pick(const double *d_A, const double *d_b, int32_t n, int32_t m, int64_t ld,
             int32_t rule, int32_t sticky, spx_state *d_state, double *d_colbuf, void *stream);

/* ---- K3: recalculate_matrix(), simplex.py:149-177 ------------------------ */
/* Out-of-place dictionary pivot (the reference deep-copies, :149): reads
 * (d_Ain, d_bin), writes (d_Aout, d_bout); swaps labels rowlab[c] <-> collab[r]
 * (:152), appends (r, c) to d_trace[npiv] (may be NULL) and increments npiv.
 * No-op unless d_state->status == SPX_PIVOT.  16 B of HBM traffic per cell. */
int spx_update(const double *d_Ain, double *d_Aout, const double *d_bin, double *d_bout,
               int32_t n, int32_t m, int64_t ld, spx_state *d_state,
               const double *d_colbuf, int32_t *d_rowlab, int32_t *d_collab,
               int32_t *d_trace, void *stream);

/* ---- the loop of get_solution(), simplex.py:179-199 / :261-269 ----------- */
/* Device-side loop over ping-pong buffers (A0,b0) <-> (A1,b1); the current
 * table is in buffer (npiv & 1) where npiv is read from d_state.  Enqueues
 * pick+update pairs in chunks of `chunk` pivots with no host round trip, then
 * reads the state back; stops on a terminal status, at d_state->max_pivots
 * (SPX_CAP), or after `stop_after` further pivots (<= 0: no such limit; the status is
 * then SPX_PIVOT in classic mode and, in look-ahead mode, the already priced outcome of
 * the current table — SPX_PIVOT, or its terminal status).  d_trace is [max_pivots][2] int32 or NULL.
 * On return *h_status / *h_npiv mirror d_state.
 *
 * mode SPX_LOOP_CLASSIC: pick k, update k, pick k+1, ... on `stream`.
 * mode SPX_LOOP_LOOKAHEAD (d_work 128-byte aligned, >= spx_solve_workspace_bytes(n)): while the
 * streaming update of pivot k runs on `stream`, a high-priority side stream owned by the
 * library prices pivot k+1 from the same (old) table — the next b column, the next f /
 * phase-1 row and the next entering column are O(n+m) cells computed with the update's own
 * arithmetic — so the update kernels run back to back and pricing is off the critical path.
 * Pivot sequence and every cell are identical in both modes. */
#define SPX_LOOP_AUTO      0  /* resident if the tableau fits L2; fused if the body is >= 256 MB; else look-ahead (workspace permitting), else classic */
#define SPX_LOOP_CLASSIC   1
#define SPX_LOOP_LOOKAHEAD 2
#define SPX_LOOP_RESIDENT  3  /* ONE persistent cooperative kernel runs the whole loop (n <= 4095, both bodies in L2):
                               * every CTA prices the pivot redundantly, one grid barrier per pivot (csrc/spx_resident.cu) */
#define SPX_LOOP_FUSED     4  /* F pivots per pass: one CTA prices the next F pivots from the stored table by replaying
                               * the pending rank-1 updates on the O(n+m) cells the rules need, then ONE stream over
                               * the body applies all F — 16 B of HBM traffic per cell per F pivots (csrc/spx_fused.cu).
                               * Workspace: spx_fused_workspace_bytes(n, m).  Same pivots, same bits. */
int64_t spx_solve_workspace_bytes(int32_t n);
int64_t spx_fused_workspace_bytes(int32_t n, int32_t m);
/* One pass of the fused loop on its own: phase 0 = price `depth` pivots + stream the body once,
 * 1 = the pricing kernel only, 2 = the fused update kernel only (after a phase-1 call).  The index
 * of the buffer holding the current table travels in d_state->reserved[0] (0/1); the caller sets it
 * before the first pass.  Used by bench.py to time the two kernels separately. */
int spx_fused_pass(double *d_A0, double *d_A1, double *d_b0, double *d_b1, int32_t n, int32_t m, int64_t ld,
                   int32_t rule, int32_t depth, int32_t phase, spx_state *d_state, void *d_work,
                   int64_t work_bytes, int32_t *d_rowlab, int32_t *d_collab, int32_t *d_trace, void *stream);
int spx_solve(double *d_A0, double *d_A1, double *d_b0, double *d_b1,
              int32_t n, int32_t m, int64_t ld, int32_t rule,
              spx_state *d_state, double *d_colbuf, int32_t *d_rowlab, int32_t *d_collab,
              int32_t *d_trace, int32_t chunk, int64_t stop_after,
              int32_t mode, void *d_work, int64_t work_bytes,
              int32_t *h_status, int64_t *h_npiv, void *stream);

/* ---- find_optimum() / f(), simplex.py:48-68, generalised to m variables --- */
/* d_x[j] = b of the row labelled x_{j+1}, else 0; d_obj[0] = function[0]*x1 +
 * function[1]*x2 exactly as :49 (0 when m < 2); d_obj[1] = sum_j function[j]*x[j]
 * accumulated left to right. */
int spx_extract(const double *d_b, int32_t n, int32_t m, const int32_t *d_collab,
                const double *d_function, double *d_x, double *d_obj, void *stream);

/* ---- K4: batches of independent small LPs, one warp per LP ---------------- */
/* d_T is [B][cells] reference-flat, solved IN PLACE (final tables left in d_T).
 * Outputs (device, any may be NULL except status/npiv):
 *   d_x [B][m], d_obj [B] (function[0]*x1+function[1]*x2, simplex.py:49),
 *   d_status [B], d_npiv [B], d_rowlab [B][m], d_collab [B][n],
 *   d_trace [B][max_pivots][2], d_snap [B][max_pivots+1][cells] (the Info.table
 *   sequence of get_solution(), simplex.py:181,198: slot k = table before pivot k).
 * The LP must fit one CTA's shared memory: spx_batched_fits(n, m). */
int spx_solve_batched(double *d_T, int64_t B, int32_t n, int32_t m, int32_t rule,
                      int32_t max_pivots, double *d_x, double *d_obj,
                      int32_t *d_status, int32_t *d_npiv,
                      int32_t *d_rowlab, int32_t *d_collab,
                      int32_t *d_trace, double *d_snap, void *stream);
int64_t spx_batched_max_cells(void);
/* Host only (no device): 1 when spx_solve_batched takes an n x m LP, else 0.  With
 * cells = n*(m+1) + m: cells <= spx_batched_max_cells(), and above 96 cells (one CTA per
 * LP) the cell lookup table and the LP's two tables, x and labels fit the shared memory
 * of a CTA beside the kernel's 16 static bytes:
 *     ceil16(4*cells) + ceil16(8*(2*cells + m) + 4*(n + m))  <=  232448 - 16 bytes.
 * E.g. 72 x 136 (10,000 cells) fits; 1 x 4470 (8,941 cells) and 2 x 3228 do not. */
int32_t spx_batched_fits(int32_t n, int32_t m);

/* ---- K7: batches of independent mid-size LPs, one thread-block cluster per LP -- */
/* The whole loop of get_solution(), simplex.py:179-199 (pick_element :70-141 and
 * recalculate_matrix :143-177 inlined), for tables above spx_batched_max_cells():
 * a cluster of S CTAs solves one LP with its table in their shared memory, CTA k
 * holding body rows [k*R, k*R+R), R = ceil(n/S), and a copy of the f row; the pivot
 * row travels over distributed shared memory, two cluster barriers per pivot.
 * Arguments, outputs and results are those of spx_solve_batched, bit for bit
 * (labels start at x1..xm / y1..yn, :30-31; final tables in place in d_T; d_snap
 * slot k = the table before pivot k, :181,198; d_obj as :49).
 * Capacity: with Q = ceil(m/S), one CTA needs
 *     8*(R*(m+2) + 2*m + 1) + 4*(R + Q)  <=  230400 bytes
 * for some S in {1, 2, 4, 8, 16} (e.g. D(100,100): S = 1, D(128,256): 2,
 * D(256,512): 8, D(512,800): 16; n <= 528 at m = 800; m <= 9499).  Shape, rule, B and the non-null
 * outputs are checked before the device is touched; a device that cannot
 * co-schedule one cluster of S CTAs is an error, not a fall-back. */
int spx_solve_batched_cluster(double *d_T, int64_t B, int32_t n, int32_t m, int32_t rule,
                              int32_t max_pivots, double *d_x, double *d_obj,
                              int32_t *d_status, int32_t *d_npiv,
                              int32_t *d_rowlab, int32_t *d_collab,
                              int32_t *d_trace, double *d_snap, void *stream);
/* Host only (no device): the smallest S in {1, 2, 4, 8, 16} whose footprint above
 * fits, i.e. the cluster size K7 uses for an n x m LP unless SPX_OPT_CLUSTER_SIZE
 * forces one; 0 when the LP does not fit one cluster. */
int32_t spx_cluster_size(int32_t n, int32_t m);

/* ---- K8: batches of LPs too large for one cluster, the table in global memory -- */
/* The loop of K7 with each LP's body rows left in d_T and updated there in place:
 * a cluster of S CTAs solves one LP, CTA k owning body rows [k*R, k*R+R), R = ceil(n/S),
 * and keeping only a copy of the f row, the old pivot row, its rows' old pivot-column
 * entries and the labels in shared memory; two cluster barriers per pivot.  Arguments,
 * NULL conventions, outputs and results are those of spx_solve_batched_cluster, bit for
 * bit, for every shape either accepts.
 * Capacity: with Q = ceil(m/S), one CTA needs
 *     8*(2*m + 1 + R) + 4*(R + Q)  <=  230400 bytes
 * for some S in {1, 2, 4, 8, 16} (m <= 11519 at S = 1 and m <= 14177 at S = 16; at
 * m = 2000, n <= 15866 at S = 1 and n <= 263856 at S = 16).
 * S: SPX_OPT_CLUSTER_SIZE when set, else spx_global_cluster_size(n, m, B).  Shape, rule,
 * B, the non-null outputs, the capacity and B*S <= INT32_MAX are checked before the
 * device is touched; B = 0 returns 0; a device that cannot co-schedule one cluster of
 * S CTAs is an error, not a fall-back. */
int spx_solve_batched_global(double *d_T, int64_t B, int32_t n, int32_t m, int32_t rule,
                             int32_t max_pivots, double *d_x, double *d_obj,
                             int32_t *d_status, int32_t *d_npiv,
                             int32_t *d_rowlab, int32_t *d_collab,
                             int32_t *d_trace, double *d_snap, void *stream);
/* Host only (no device): S_min, the smallest S in {1, 2, 4, 8, 16} whose footprint
 * above fits; 0 when the LP does not fit. */
int32_t spx_global_min_cluster_size(int32_t n, int32_t m);
/* The S a K8 solve of B such LPs launches on the current device: SPX_OPT_CLUSTER_SIZE
 * when set (0 if it does not fit); else the S >= S_min that keeps the most SMs busy,
 * min(B, cudaOccupancyMaxActiveClusters at S) * S, the smaller S on ties, so a single LP
 * gets 16 CTAs and a batch that fills the device at S_min gets S_min; 0 when the LP does
 * not fit, -1 on a CUDA error.  Queries occupancy, launches nothing. */
int32_t spx_global_cluster_size(int32_t n, int32_t m, int64_t B);

/* ---- ragged batches: LPs of any mix of shapes in one call (K4, K7 and K8) ------- */
/* Each LP k has its own shape (n_k, m_k) and its own cap max_pivots_k.  Every buffer
 * is packed in batch order: LP k's slice starts at the prefix sum over LPs 0..k-1 of
 *     d_T, d_snap-table   cells          d_x, d_rowlab   m
 *     d_collab            n              d_trace         max_pivots (pairs of int32)
 *     d_snap              (max_pivots+1)*cells
 * and d_obj, d_status, d_npiv hold one element per LP.  Each LP's results are those
 * of spx_solve_batched / spx_solve_batched_cluster / spx_solve_batched_global for that
 * LP alone, bit for bit.
 *
 * Routing: each LP goes where spx_batched_route sends it, K7 at spx_cluster_size(n, m)
 * or SPX_OPT_CLUSTER_SIZE when set.  One solve makes at most 12 launches, in
 * sequence on `stream`: K4 warp mode (LPs of <= 96 cells) if any, K4 CTA mode if any,
 * one K7 launch per distinct cluster size, then one K8 launch per distinct S_min
 * (spx_global_min_cluster_size), or one at SPX_OPT_CLUSTER_SIZE when it is set when the
 * plan is made.  Within a launch the LPs run largest first (by cells, ties by batch
 * index).  A K8 launch planned without SPX_OPT_CLUSTER_SIZE runs at the S that
 * spx_ragged_cluster_size reports: the rule of spx_global_cluster_size applied to the
 * launch, over S >= its S_min, with the largest footprint of its LPs at each S. */
#define SPX_ENGINE_AUTO        0
#define SPX_ENGINE_SMEM        1
#define SPX_ENGINE_CLUSTER     2
#define SPX_ENGINE_GLOBAL      4
#define SPX_ENGINE_AUTO_GLOBAL 5
/* Host only (no device): the engine that takes an n x m LP under `engine`, the rule of
 * spx_ragged_plan and of the uniform entries: SPX_ENGINE_SMEM (K4), SPX_ENGINE_CLUSTER
 * (K7) or SPX_ENGINE_GLOBAL (K8).  SPX_ENGINE_AUTO sends an LP to K4 when
 * spx_batched_fits(n, m), else to K7, and rejects an LP above K7's capacity
 * (spx_cluster_size(n, m) == 0); SMEM, CLUSTER and GLOBAL send every LP to that engine;
 * AUTO_GLOBAL is AUTO with K8 for the LPs above K7's capacity, up to K8's.  Code 3 is
 * not an engine.  -1 when the engine cannot take the LP (spx_last_error() names the
 * capacity it exceeds), the shape is not n, m >= 1, or the code is unknown.
 * SPX_OPT_CLUSTER_SIZE is not read: the plan and the uniform entries also refuse an LP
 * that does not fit the cluster size it forces. */
int32_t spx_batched_route(int32_t n, int32_t m, int32_t engine);
/* bytes of the plan of a batch of B LPs (-1 when B < 0) */
int64_t spx_ragged_plan_bytes(int64_t B);
/* Host only, no device.  h_shapes[B][3] = {n, m, max_pivots} in batch order.  Validates
 * every LP (the error text names the first bad LP's index and the capacity it exceeds),
 * reads SPX_OPT_CLUSTER_SIZE, and writes into h_plan (plan_bytes >= spx_ragged_plan_bytes(B))
 * the per-LP descriptors (shape and offsets above) and the launch list (kernel, cluster
 * size, block size, dynamic shared memory, the LP indices largest first).
 * h_totals[5] = the packed lengths of T, x (= rowlab), collab, trace (pairs) and snap. */
int spx_ragged_plan(const int32_t *h_shapes, int64_t B, int32_t engine, void *h_plan, int64_t plan_bytes,
                    int64_t *h_totals);
/* Solves the batch h_plan describes.  d_plan is a byte copy of h_plan in device memory,
 * made by the caller (nothing allocates behind the caller's back and there is no hidden
 * synchronising copy).  The launches are read from h_plan, the descriptors from d_plan.
 * Plan header, rule and pointers are checked before the device is touched; a plan of
 * B = 0 returns 0.  Outputs and NULL conventions as spx_solve_batched.  A K8 launch
 * checks count * S <= INT32_MAX for the S it launches at; a device that cannot
 * co-schedule one of its clusters is an error naming S and the footprint. */
int spx_solve_batched_ragged(double *d_T, const void *h_plan, const void *d_plan, int32_t rule,
                             double *d_x, double *d_obj, int32_t *d_status, int32_t *d_npiv,
                             int32_t *d_rowlab, int32_t *d_collab, int32_t *d_trace, double *d_snap,
                             void *stream);
/* The cluster size launch `launch` (0-based) of h_plan runs at on the current device: the
 * planned S for K4 (1) and K7, and for K8 the planned S when SPX_OPT_CLUSTER_SIZE was set
 * at plan time (no device needed), else the rule above (queries occupancy, launches
 * nothing).  -1 on error. */
int32_t spx_ragged_cluster_size(const void *h_plan, int32_t launch);

/* ---- sensitivity report of optimal final tables (csrc/spx_sensitivity.cu) ------- */
/* The final table is a dictionary: x_B = b + T x_N, f = f0 + sum_j d_j x_N (recalculate_matrix,
 * :143-177); the LP is: minimise c.x subject to b + A x >= 0, x >= 0.  Constraint k's slack is y_k.
 * Per constraint k (n of each; ranges are [n][2] = (allowable decrease, allowable increase)):
 *   y_k nonbasic in column j: dual = -d_j, slack = 0, rhs_range = (min over rows i with T[i][j] < 0
 *                             of b_i / (-T[i][j]), min over rows with T[i][j] > 0 of b_i / T[i][j]);
 *   y_k basic in row i:       dual = 0, slack = b_i, rhs_range = (b_i, +inf).
 * Per variable k (m of each):
 *   x_k nonbasic in column j: reduced_cost = d_j, cost_range = (d_j, +inf);
 *   x_k basic in row i:       reduced_cost = 0, cost_range = (min over columns j with T[i][j] > 0 of
 *                             d_j / T[i][j], min over columns with T[i][j] < 0 of d_j / (-T[i][j])).
 * Each quotient is one IEEE division; a minimum over an empty set is +inf, a NaN quotient never
 * wins, every zero is written as +0.0, and every output of an LP that is not optimal is NaN.  A
 * minimum does not depend on the order of reduction, so the results equal a sequential statement
 * bit for bit.  Labels and status are required; each output pointer may be NULL.  Arguments and
 * shapes (and the plan header) are checked before the device is touched; B = 0 returns 0.
 *
 * Uniform batches: d_T [B][cells] final reference-flat tables (DeviceBatch after K4, K7 or K8),
 * d_status [B], d_rowlab [B][m], d_collab [B][n]; d_dual, d_slack [B][n], d_rhs_range [B][n][2],
 * d_redcost [B][m], d_cost_range [B][m][2].  An LP is optimal when d_status[k] == SPX_OPTIMAL. */
int spx_sensitivity_batched(const double *d_T, int64_t B, int32_t n, int32_t m, const int32_t *d_status,
                            const int32_t *d_rowlab, const int32_t *d_collab, double *d_dual, double *d_slack,
                            double *d_redcost, double *d_rhs_range, double *d_cost_range, void *stream);
/* Ragged batches packed as spx_solve_batched_ragged packs them: per-constraint outputs at the prefix
 * sums of n (as d_collab; ranges twice that), per-variable outputs at the prefix sums of m (as d_x). */
int spx_sensitivity_ragged(const double *d_T, const void *h_plan, const void *d_plan, const int32_t *d_status,
                           const int32_t *d_rowlab, const int32_t *d_collab, double *d_dual, double *d_slack,
                           double *d_redcost, double *d_rhs_range, double *d_cost_range, void *stream);
/* One split table (d_A [(n+1)][ld], d_b [n]; d_rowlab [m], d_collab [n]), e.g. the current table of
 * a streaming solve.  Optimality is decided from the table with pick_element's tests (:72-76 and
 * :94-98: no b cell and no f cell negative), which copies b and the f row to the host and
 * synchronises `stream`; *h_optimal = 1 when optimal, else 0 and every output is NaN. */
int spx_sensitivity_split(const double *d_A, const double *d_b, int32_t n, int32_t m, int64_t ld,
                          const int32_t *d_rowlab, const int32_t *d_collab, double *d_dual, double *d_slack,
                          double *d_redcost, double *d_rhs_range, double *d_cost_range, int32_t *h_optimal,
                          void *stream);

/* ---- certificates of infeasible and unbounded LPs (csrc/spx_certificate.cu) ------- */
/* Conventions of the sensitivity report above: label codes x_k -> k, y_k -> m + k, rowlab [m] over the columns,
 * collab [n] over the rows, w1 = m + 1, b_i = T[i*w1 + m], d_j = T[n*w1 + j].  Computed for every LP from its final
 * table, whatever its status, in this sequential statement:
 *   Farkas row:  farkas_row = the lowest i with b_i finite and < 0 and every T[i][j] (j < m) finite and <= 0, else -1.
 *                Found: farkas [n] = +0.0 everywhere; then farkas[L-m] = 1.0 when L = collab[r] is a y label; then,
 *                for j ascending, farkas[H-m] = 0.0 - T[r][j] when H = rowlab[j] is a y label (+0.0 for either zero);
 *                farkas_bound = b_r.  Not found: farkas all NaN, farkas_bound NaN.
 *   Ray column:  only when every b_i is finite and >= 0 (-0.0 counts): ray_col = the lowest j with d_j finite and < 0
 *                and every T[i][j] (i < n) finite and >= 0, else -1.
 *                Found: ray [m] = +0.0 everywhere; then ray[H] = 1.0 when H = rowlab[c] is an x label; then, for i
 *                ascending, ray[L] = T[i][c] + 0.0 when L = collab[i] is an x label; ray_slope = d_c.  Not found:
 *                ray all NaN, ray_slope NaN.
 * A label outside its range is skipped.  Why they are certificates, for "minimise c.x subject to b + A x >= 0,
 * x >= 0": row r says a non-negative variable equals b_r < 0 plus a non-positive combination of non-negative ones,
 * so u = farkas >= 0 has A^T u <= 0 and b.u = b_r < 0 (the LP is infeasible); in a table with b >= 0, raising x_N_c
 * from the vertex keeps every constraint and lowers f by |d_c| per unit, so d = ray >= 0 has A d >= 0 and
 * c.d = d_c < 0 (the LP is unbounded).  An SPX_INCORRECT table gets the row the solver stopped on; an SPX_NOCONV
 * table of the reference rule gets the solver's entering column; an optimal table gets neither.  Every step is a
 * minimum of indices, a logical OR or a copy, so the results equal the statement bit for bit.
 *
 * Outputs: d_row [B] int32, d_farkas, d_bound [B], d_col [B] int32, d_ray, d_slope [B].  Each may be NULL, with one
 * rule: d_farkas and d_ray are the kernels' only workspace (no memory is allocated), so d_row and d_bound need
 * d_farkas, and d_col and d_slope need d_ray.  Labels are required.  Arguments, shapes and the plan header are
 * checked before the device is touched; B = 0 returns 0.  At most three launches per group, no synchronisation.
 *
 * Uniform batches: d_T [B][cells] final reference-flat tables (DeviceBatch after K4, K7 or K8), d_rowlab [B][m],
 * d_collab [B][n]; d_farkas [B][n], d_ray [B][m]. */
int spx_certificate_batched(const double *d_T, int64_t B, int32_t n, int32_t m, const int32_t *d_rowlab,
                            const int32_t *d_collab, int32_t *d_row, double *d_farkas, double *d_bound,
                            int32_t *d_col, double *d_ray, double *d_slope, void *stream);
/* Ragged batches packed as spx_solve_batched_ragged packs them, one group of launches per launch of the plan:
 * d_farkas at the prefix sums of n (as d_collab), d_ray at those of m (as d_x); the per-LP outputs [B]. */
int spx_certificate_ragged(const double *d_T, const void *h_plan, const void *d_plan, const int32_t *d_rowlab,
                           const int32_t *d_collab, int32_t *d_row, double *d_farkas, double *d_bound,
                           int32_t *d_col, double *d_ray, double *d_slope, void *stream);
/* One split table (d_A [(n+1)][ld], d_b [n]; d_rowlab [m], d_collab [n]), e.g. the current table of a streaming
 * solve; the per-LP outputs have one element. */
int spx_certificate_split(const double *d_A, const double *d_b, int32_t n, int32_t m, int64_t ld,
                          const int32_t *d_rowlab, const int32_t *d_collab, int32_t *d_row, double *d_farkas,
                          double *d_bound, int32_t *d_col, double *d_ray, double *d_slope, void *stream);

/* ---- warm start: change and resume final tables (csrc/spx_warm.cu) ---------------- */
/* The final table of a batched solve is a dictionary (conventions of the sensitivity report above;
 * label codes x_k -> k, y_k -> m + k, w1 = m + 1, b_i = T[i*w1 + m], d_j = T[n*w1 + j]).  The change
 * entries apply new right-hand sides b + db and costs c + dc to final tables IN PLACE, per LP and in
 * exactly this order (every product and sum rounded on its own, no FMA; the body cells are never
 * written):
 *   for each row i in [0, n):      v = b_i;  L = collab[i];  if m <= L < m+n and db[L-m] != 0: v = v + db[L-m];
 *                                  for j = 0 .. m-1 ascending: H = rowlab[j];
 *                                      if m <= H < m+n and (d = db[H-m]) != 0: v = v - d*T[i][j];
 *                                  b_i = v
 *   for each column j in [0, m):   v = d_j;  H = rowlab[j];  if 0 <= H < m and dc[H] != 0: v = v + dc[H];
 *                                  for i = 0 .. n-1 ascending: L = collab[i];
 *                                      if 0 <= L < m and (d = dc[L]) != 0: v = v + d*T[i][j];
 *                                  d_j = v
 * A zero delta (-0.0 included) leaves the table bit for bit; a label outside its range is skipped.  The
 * b update reads only body columns j < m and the f update only body rows, so both run in one launch.
 * Uniform: d_T [B][cells], d_rowlab [B][m], d_collab [B][n], d_delta_b [B][n], d_delta_c [B][m].  Ragged
 * (packed as spx_solve_batched_ragged): d_delta_b at the prefix sums of n (as d_collab), d_delta_c at
 * those of m (as d_x).  Either delta may be NULL; with both NULL, or B = 0, nothing is done and 0 is
 * returned.  Labels are required.  Arguments (and the plan header) are checked before the device is
 * touched.  No workspace. */
int spx_warm_change_batched(double *d_T, int64_t B, int32_t n, int32_t m, const int32_t *d_rowlab,
                            const int32_t *d_collab, const double *d_delta_b, const double *d_delta_c, void *stream);
int spx_warm_change_ragged(double *d_T, const void *h_plan, const void *d_plan, const int32_t *d_rowlab,
                           const int32_t *d_collab, const double *d_delta_b, const double *d_delta_c, void *stream);
/* Continue every LP for up to max_pivots (ragged: the plan's caps) more pivots from the table in d_T and
 * the labels in d_rowlab / d_collab, which are required and in/out; the pivot loop is that of the solve
 * entries, and the trace and snapshots count from 0 in each call.  Uniform: engine as spx_batched_route
 * (AUTO, SMEM, CLUSTER, GLOBAL, AUTO_GLOBAL) with the routing, cluster-size rules and SPX_OPT_CLUSTER_SIZE
 * of spx_solve_batched / _cluster / _global; a resume may run on another engine or cluster size than the
 * solve before it and computes the same bits.  d_function ([B][m], ragged packed as d_x) holds the LPs'
 * current costs, used only for d_obj = function[0]*x1 + function[1]*x2; required when d_obj != NULL.
 * Outputs, NULL conventions and errors otherwise as spx_solve_batched / spx_solve_batched_ragged; B = 0
 * returns 0. */
int spx_warm_solve_batched(int32_t engine, double *d_T, int64_t B, int32_t n, int32_t m, int32_t rule,
                           int32_t max_pivots, const double *d_function, double *d_x, double *d_obj,
                           int32_t *d_status, int32_t *d_npiv, int32_t *d_rowlab, int32_t *d_collab,
                           int32_t *d_trace, double *d_snap, void *stream);
int spx_warm_solve_ragged(double *d_T, const void *h_plan, const void *d_plan, int32_t rule,
                          const double *d_function, double *d_x, double *d_obj, int32_t *d_status,
                          int32_t *d_npiv, int32_t *d_rowlab, int32_t *d_collab, int32_t *d_trace,
                          double *d_snap, void *stream);

/* ---- column-sharded large tableau (one process per GPU) ------------------- */
/* Rank g owns global columns [col0, col0+m_loc) of the body as a local split
 * matrix d_A[(n+1)][ld_loc]; b, the labels and the state are replicated.  Per pivot:
 *   spx_shard_candidate : local K1 — this shard's best entering column (key;
 *                         none = all ones) and that column's n+1 cells, packed
 *                         into d_send = [header | column], spx_shard_msg_doubles(n)
 *                         doubles;
 *   (all-gather of d_send over NCCL/NVLink — done by the caller)
 *   spx_shard_select    : global K1 (min key over ranks) + K2 ratio test on the
 *                         winning column with the replicated b; writes d_state
 *                         (c is GLOBAL) and d_colbuf;
 *   spx_shard_update    : K3 on the local columns; every rank updates its b.
 * With nranks == 1 the three calls reproduce spx_pick + spx_update exactly. */
int64_t spx_shard_msg_doubles(int32_t n);
int spx_shard_candidate(const double *d_A, const double *d_b, int32_t n, int32_t m_loc,
                        int64_t ld_loc, int64_t col0, int32_t rule, int32_t sticky,
                        spx_state *d_state, double *d_send, void *stream);
/* d_flags/seq: NULL/0 after a library all-gather; with peer mailboxes (below) the LOCAL flag
 * words flags[parity][nranks] and the exchange number to wait for. */
int spx_shard_select(const double *d_gathered, int32_t nranks, const double *d_b,
                     int32_t n, int32_t rule, int32_t sticky, spx_state *d_state,
                     double *d_colbuf, const uint64_t *d_flags, uint64_t seq, void *stream);
/* ahead != 0: look-ahead mode — the kernel only reads *d_state, skips the b column and the
 * pricing hints (spx_ahead_candidate / spx_ahead_select own them) and still swaps the labels
 * and appends to the trace. */
int spx_shard_update(const double *d_Ain, double *d_Aout, const double *d_bin, double *d_bout,
                     int32_t n, int32_t m_loc, int64_t ld_loc, int64_t col0,
                     spx_state *d_state, const double *d_colbuf,
                     int32_t *d_rowlab, int32_t *d_collab, int32_t *d_trace,
                     int32_t ahead, void *stream);

/* Look-ahead halves of the sharded flow: they price pivot k+1 from table k (the table the
 * running update of pivot k reads), so they can run on another stream concurrently with it:
 *   spx_ahead_candidate : next b column (d_bin -> d_bout, every rank), this shard's best
 *                         entering column of the NEXT table and that column's n+1 next cells,
 *                         packed into d_send (spx_shard_msg_doubles(n) doubles);
 *   (all-gather of d_send)
 *   spx_ahead_select    : min key over ranks + ratio test with the next b; writes the NEXT
 *                         state (npiv+1) and colbuf, leaving the current ones untouched.
 * Terminal states propagate: once *d_state_cur is not SPX_PIVOT the next state is a copy. */
int spx_ahead_candidate(const double *d_A, const double *d_bin, double *d_bout, int32_t n, int32_t m_loc,
                        int64_t ld_loc, int64_t col0, int32_t rule, const spx_state *d_state,
                        const double *d_colbuf, double *d_send, void *stream);
int spx_ahead_select(const double *d_gathered, int32_t nranks, const double *d_bnext, int32_t n,
                     const spx_state *d_state_cur, spx_state *d_state_next, double *d_colbuf_next,
                     const uint64_t *d_flags, uint64_t seq, void *stream);

/* ---- the exchange over NVLink peer memory (no library collective on the data path) -------
 * Each rank owns a MAILBOX  gathered[2][nranks][spx_shard_msg_doubles(n)] | flags[2][nranks]
 * (spx_mailbox_bytes, zero-initialised, allocated with spx_device_alloc so that it can be
 * exported over CUDA IPC to the other ranks' processes).  spx_peer_push stores this rank's
 * message into EVERY rank's mailbox (one CTA per destination, 128-bit stores through NVLink)
 * and release-stores `seq` into the destination's flag word; the select kernels acquire-poll
 * their local flags (20 s timeout -> SPX_PEER_TIMEOUT).  parity = seq & 1. */
typedef struct spx_shard spx_shard;
int     spx_device_alloc(void **d_ptr, int64_t bytes);
int     spx_device_free(void *d_ptr);
int     spx_ipc_handle_bytes(void);
int     spx_ipc_export(void *d_ptr, void *handle_out);
int     spx_ipc_import(const void *handle, void **d_ptr);
int     spx_ipc_close(void *d_ptr);
int64_t spx_mailbox_bytes(int32_t n, int32_t nranks);
int     spx_peer_push(const double *d_send, int32_t n, int32_t rank, int32_t nranks, int32_t parity,
                      uint64_t seq, void *const *mailboxes, void *stream);

/* The whole sharded look-ahead loop behind one handle, enqueued from C (no Python and no
 * collective library per pivot): spx_shard_enqueue(h, K) enqueues K pivots — update k on
 * `stream`, pricing of pivot k+1 (next b, local candidate, peer push, select) on the handle's
 * high-priority side stream — and returns; every rank must enqueue the same K.
 *   d_state2  : spx_state[2] (element 0 initialised by spx_init_state)
 *   d_colbuf2 : 2 * spx_colbuf_doubles(n) doubles
 *   mailboxes : nranks device pointers valid in THIS process ([rank] = the local mailbox)
 * spx_shard_read synchronises `stream`, returns the current (already priced) state and the
 * index (0/1) of the ping-pong buffer that holds the current table. */
int spx_shard_open(spx_shard **out, int32_t rank, int32_t nranks, int32_t n, int32_t m_loc, int64_t ld_loc,
                   int64_t col0, int32_t rule, double *d_A0, double *d_A1, double *d_b0, double *d_b1,
                   spx_state *d_state2, double *d_colbuf2, int32_t *d_rowlab, int32_t *d_collab,
                   int32_t *d_trace, double *d_send, void *const *mailboxes);
int spx_shard_reset(spx_shard *h);
int spx_shard_enqueue(spx_shard *h, int64_t pivots, void *stream);
int spx_shard_read(spx_shard *h, spx_state *h_state, int32_t *cur_buffer, void *stream);
int spx_shard_close(spx_shard *h);

/* ---- the column-sharded FUSED loop (one process per GPU, csrc/spx_fused.cu) -------------------
 * Passes of `depth` pivots: a whole-GPU cooperative kernel on every rank prices the next pivots by
 * lazy replay and exchanges, per pivot and from INSIDE the kernel over NVLink peer memory, the
 * ranks' 16-byte entering-column keys and the winning pivot column (stored by its owner straight
 * into every rank's plane); then each rank streams its own columns once and applies all pivots.
 * Each rank owns an XBOX (spx_fshard_xbox_bytes, zero-initialised, spx_device_alloc + CUDA IPC);
 * `xboxes` lists every rank's XBOX as mapped into this process.  d_state->reserved[0] carries the
 * index of the ping-pong buffer that holds the current table (0 after spx_init_state);
 * spx_fshard_read returns it.  d_work: spx_fused_workspace_bytes(n, m_loc) bytes. */
typedef struct spx_fshard spx_fshard;
int64_t spx_fshard_xbox_bytes(int32_t n, int32_t nranks);
int spx_fshard_open(spx_fshard **out, int32_t rank, int32_t nranks, int32_t n, int32_t m_loc, int64_t ld_loc,
                    int64_t col0, int32_t rule, double *d_A0, double *d_A1, double *d_b0, double *d_b1,
                    spx_state *d_state, void *d_work, int64_t work_bytes, int32_t *d_rowlab, int32_t *d_collab,
                    int32_t *d_trace, void *const *xboxes);
/* look-ahead (default 1): the pricing of pass q+1 runs on the handle's high-priority side stream while
 * the update of pass q streams; 0: price, update, price, ... on `stream`; 2: look-ahead with a PERSISTENT
 * pricing engine — one cooperative pricing kernel per spx_fshard_enqueue call prices every pass and keeps its
 * SMs, the update kernels of all passes are enqueued behind it at once, and the two dependencies (update q
 * needs plan q; pricing q needs the table of update q-2) go through device flags instead of one cooperative
 * launch and two events per pass.  Opt-in: measured no faster than mode 1 on cfg4 (8 ranks 19.5 k vs 19.3 k pivots/s,
 * 2 ranks 6.4 k vs 7.0 k).  Every rank must use the same mode. */
int spx_fshard_set_lookahead(spx_fshard *h, int32_t on);
int spx_fshard_enqueue(spx_fshard *h, int64_t pivots, int32_t depth, void *stream);
int spx_fshard_read(spx_fshard *h, spx_state *h_state, int32_t *cur_buffer, void *stream);
int spx_fshard_close(spx_fshard *h);
/* Developer aid: the %globaltimer stamps (ns) the sharded pricing kernel left in the fused workspace `d_work` during
 * its LAST launch: h_out[9][6] = per level {phase A done, entering column known (grid barrier 1), candidate columns
 * stored on every rank, keys exchanged over NVLink, ratio partials in (grid barrier 2), level recorded}.
 * Synchronises `stream`.  No reference counterpart. */
int spx_fused_debug_stamps(const void *d_work, int32_t n, int64_t ld, uint64_t *h_out, int32_t capacity, void *stream);
/* Developer aid: with SPX_RESIDENT_STAMPS=1 in the environment the L2-resident persistent kernel accumulates clock64()
 * cycles per phase of a pivot (thread 0 of CTA 0); h_out16[0..14] = the sums over the last launch in the order of the
 * kernel's pc.mark(k) calls (csrc/spx_resident.cu), h_out16[15] = pivots applied.  No reference counterpart. */
int spx_resident_debug(uint64_t *h_out16);

#ifdef __cplusplus
}
#endif
#endif /* SPX_B200_H */
