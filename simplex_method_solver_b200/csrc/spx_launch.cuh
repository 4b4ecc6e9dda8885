// spx_launch.cuh — the host launchers and queries the .cu files define for the C entries of spx_api.cu.  Every file that
// defines one includes this header, so the compiler checks each definition against its declaration.
#pragma once
#include "spx_common.cuh"

namespace spx_launch {

// ---- options and device (spx_update.cu) ----
int     sm_count();
int64_t get_option(int key);
int     set_option(int key, int64_t value);

// ---- K1 + K2 (spx_pick.cu), K3 (spx_update.cu) and the split loop's helpers ----
int64_t colbuf_doubles(int n);
int64_t shard_msg_doubles(int n);
cudaError_t pick(const double *A, const double *b, int n, int m, int64_t ld, int rule, int sticky, spx_state *st,
                 double *colbuf, cudaStream_t stream);
cudaError_t shard_candidate(const double *A, const double *b, int n, int m_loc, int64_t ld, int64_t col0, int rule,
                            int sticky, const spx_state *st, double *msg, cudaStream_t stream);
cudaError_t shard_select(const double *gathered, int nranks, const double *b, int n, int sticky, spx_state *st,
                         double *colbuf, const unsigned long long *flags, unsigned long long seq, cudaStream_t stream);
cudaError_t ahead_candidate(const double *A, const double *bin, double *bout, int n, int m_loc, int64_t ld,
                            int64_t col0, int rule, const spx_state *st, const double *colbuf, double *msg,
                            cudaStream_t stream);
cudaError_t ahead_select(const double *gathered, int nranks, const double *bnext, int n, const spx_state *st_cur,
                         spx_state *st_next, double *colbuf_next, const unsigned long long *flags,
                         unsigned long long seq, cudaStream_t stream);
cudaError_t update(const double *Ain, double *Aout, const double *bin, double *bout, int n, int m_loc, int64_t ld,
                   int64_t col0, spx_state *st, const double *colbuf, int32_t *rowlab, int32_t *collab,
                   int32_t *trace, int ahead, cudaStream_t stream);
cudaError_t extract(const double *b, int n, int m, const int32_t *collab, const double *function, double *x,
                    double *obj, cudaStream_t stream);
cudaError_t init_state(spx_state *st, int32_t *rowlab, int32_t *collab, int n, int m, int64_t max_pivots,
                       cudaStream_t stream);
cudaError_t selftest_division(const double *a, const double *p, int64_t count, int64_t np,
                              unsigned long long *d_mismatches, double *d_first_bad, cudaStream_t stream);

// ---- the L2-resident loop (spx_resident.cu) and the fused loop (spx_fused.cu) ----
bool resident_fits(int n, int m, int64_t ld);
cudaError_t resident_loop(double *A0, double *A1, double *b0, double *b1, int n, int m, int64_t ld, int rule,
                          int64_t max_steps, spx_state *st, double *colbuf, int32_t *rowlab, int32_t *collab,
                          int32_t *trace, cudaStream_t stream);
int fuse_max();                 // levels per pass at most of the one-GPU fused loop
int64_t fused_workspace_bytes(int n, int64_t ld);
cudaError_t fused_pass(double *A0, double *A1, double *b0, double *b1, int n, int m, int64_t ld, int rule, int F,
                       int minb, int pricing, int phase, spx_state *st, void *work, int32_t *rowlab, int32_t *collab,
                       int32_t *trace, cudaStream_t stream);
cudaError_t fused_solve_passes(double *A0, double *A1, double *b0, double *b1, int n, int m, int64_t ld, int rule,
                               spx_state *st, void *work, int32_t *rowlab, int32_t *collab, int32_t *trace,
                               int64_t pivots, int depth, int minb, int engine, cudaStream_t s);
cudaError_t fused_solo_sync();
cudaError_t lazy_guard_selftest(const double *t0, const double *p, const double *rj, const double *ci, int F,
                                int64_t count, double *out_lazy, double *out_ref, unsigned long long *n_redo,
                                cudaStream_t stream);
cudaError_t two_op_selftest(const double *p, int64_t np, int64_t per_p, int32_t *flags, unsigned long long *mismatches,
                            cudaStream_t stream);

// ---- batched engines: K4 (spx_batched.cu), K7 (spx_cluster.cu), K8 (spx_global.cu) ----
// The uniform launchers solve B LPs of one n x m shape; the ragged launchers run launch l of plan v.  Each returns
// the launch's error; K7 and K8 return cudaErrorInvalidClusterSize when the device cannot co-schedule one cluster.
int64_t batched_max_cells();
bool batched_fits(int n, int m);
cudaError_t solve_batched(int64_t B, int n, int m, int max_pivots, const spx::BatchIO &io, cudaStream_t stream);
int64_t ragged_batched_bytes(int n, int m, int *kernel);
int ragged_cta_threads(int64_t cells);
int ragged_warps_per_cta(int64_t slot, int64_t count);
cudaError_t solve_ragged_batched(const spx::PlanView &v, const spx::RaggedLaunch &l, const spx::BatchIO &io,
                                 cudaStream_t stream);

bool cluster_fits(int64_t n, int64_t m, int S);
int cluster_size(int64_t n, int64_t m);
cudaError_t solve_batched_cluster(int64_t B, int n, int m, int S, int max_pivots, const spx::BatchIO &io,
                                  cudaStream_t stream);
int64_t ragged_cluster_bytes(int n, int m, int S);
cudaError_t solve_ragged_cluster(const spx::PlanView &v, const spx::RaggedLaunch &l, const spx::BatchIO &io,
                                 cudaStream_t stream);

bool global_fits(int64_t n, int64_t m, int S);
int global_min_cluster_size(int64_t n, int64_t m);
cudaError_t global_cluster_size(int64_t n, int64_t m, int64_t B, int *S_out);
cudaError_t solve_batched_global(int64_t B, int n, int m, int S, int max_pivots, const spx::BatchIO &io,
                                 cudaStream_t stream);
int64_t ragged_global_bytes(int n, int m, int S);
cudaError_t ragged_global_size(const spx::PlanView &v, const spx::RaggedLaunch &l, int *S_out, int64_t *smem_out);
cudaError_t solve_ragged_global(const spx::PlanView &v, const spx::RaggedLaunch &l, int S, int64_t smem,
                                const spx::BatchIO &io, cudaStream_t stream);

// ---- sensitivity report (spx_sensitivity.cu) and warm start (spx_warm.cu) ----
cudaError_t sensitivity_uniform(const double *d_T, int64_t B, int n, int m, const int32_t *d_status,
                                const int32_t *d_rowlab, const int32_t *d_collab, double *dual, double *slack,
                                double *redcost, double *rhs, double *cost, cudaStream_t s);
cudaError_t sensitivity_ragged(const spx::PlanView &v, const double *d_T, const int32_t *d_status,
                               const int32_t *d_rowlab, const int32_t *d_collab, double *dual, double *slack,
                               double *redcost, double *rhs, double *cost, cudaStream_t s);
cudaError_t sensitivity_split(const double *d_A, const double *d_b, int n, int m, int64_t ld, int optimal,
                              const int32_t *d_rowlab, const int32_t *d_collab, double *dual, double *slack,
                              double *redcost, double *rhs, double *cost, cudaStream_t s);
// ---- certificates of infeasible and unbounded LPs (spx_certificate.cu) ----
cudaError_t certificate_uniform(const double *d_T, int64_t B, int n, int m, const int32_t *d_rowlab,
                                const int32_t *d_collab, int32_t *row, double *farkas, double *bound, int32_t *col,
                                double *ray, double *slope, cudaStream_t s);
cudaError_t certificate_ragged(const spx::PlanView &v, const double *d_T, const int32_t *d_rowlab,
                               const int32_t *d_collab, int32_t *row, double *farkas, double *bound, int32_t *col,
                               double *ray, double *slope, cudaStream_t s);
cudaError_t certificate_split(const double *d_A, const double *d_b, int n, int m, int64_t ld,
                              const int32_t *d_rowlab, const int32_t *d_collab, int32_t *row, double *farkas,
                              double *bound, int32_t *col, double *ray, double *slope, cudaStream_t s);
cudaError_t warm_change_uniform(double *T, int64_t B, int n, int m, const int32_t *rowlab, const int32_t *collab,
                                const double *db, const double *dc, cudaStream_t s);
cudaError_t warm_change_ragged(const spx::PlanView &v, double *T, const int32_t *rowlab, const int32_t *collab,
                               const double *db, const double *dc, cudaStream_t s);

} // namespace spx_launch
