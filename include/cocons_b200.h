/* cocons_b200 - C ABI of the B200-native dense-likelihood path of blasif/cocons.
 *
 * Everything here is `extern "C"`, plain pointers and sizes.  Matrices are
 * column-major IEEE doubles, exactly as R holds them; `theta6` is six
 * length-p vectors back to back in the order
 *     std.dev, scale, aniso, tilt, smooth, nugget
 * i.e. the named list the reference looks up at src/cocons_full.cpp:47-54
 * (the R glue in cocons_b200/rglue/cocons_glue.c does that lookup by name).
 *
 * Status codes: 0 ok; k > 0 the leading minor of order k is not positive
 * definite (LAPACK dpotrf convention - the caller maps it to the reference's
 * `tryCatch(chol(...))` logic, R/neg2loglikelihood.R:200-206); < 0 a
 * CUDA/NCCL/argument error, text in cocons_last_error().
 *
 * There is no CPU fallback: every entry point that computes fails with
 * COCONS_ERR_NO_DEVICE when no sm_100 device is usable.  The stateless and
 * one-shot entry points run on device $COCONS_DEVICE (default 0).
 */
#ifndef COCONS_B200_H
#define COCONS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COCONS_ERR_ARG (-1)
#define COCONS_ERR_CUDA (-2)
#define COCONS_ERR_NO_DEVICE (-3)
#define COCONS_ERR_ALLOC (-4)
#define COCONS_ERR_STATE (-5)

/* objective kinds for cocons_n2ll() */
#define COCONS_ML 0      /* GetNeg2loglikelihood        R/neg2loglikelihood.R:183-222 */
#define COCONS_PROFILE 1 /* GetNeg2loglikelihoodProfile R/neg2loglikelihood.R:127-165 */
#define COCONS_REML 2    /* GetNeg2loglikelihoodREML    R/neg2loglikelihood.R:241-291 */

/* covariance parameterisations */
#define COCONS_PAR_DIFF 0    /* cov_rns          src/cocons_full.cpp:40-321  */
#define COCONS_PAR_CLASSIC 1 /* cov_rns_classic  src/cocons_full.cpp:480-594 */

typedef struct cocons_ctx cocons_ctx;

/* ---- library ---------------------------------------------------------- */
int cocons_version(void);
const char* cocons_last_error(void);
int cocons_device_count(void);
/* kernels launched by this process so far (bench.py's gpu_launches) */
long long cocons_launch_count(void);

/* ---- stateless covariance builders, host buffers in and out ------------ */

/* Replaces `_cocons_cov_rns` (src/RcppExports.cpp:29-40 -> cov_rns,
 * src/cocons_full.cpp:40-321).  out: n x n, full symmetric. */
int cocons_cov_rns(int64_t n, int64_t p, const double* locs, const double* x_covariates, const double* theta6,
                   const double* smooth_limits, double* out);

/* Replaces `_cocons_cov_rns_pred` (src/RcppExports.cpp:43-56 -> cov_rns_pred,
 * src/cocons_full.cpp:334-471).  out: m x n, prediction sites are rows. */
int cocons_cov_rns_pred(int64_t n, int64_t m, int64_t p, const double* locs, const double* locs_pred,
                        const double* x_covariates, const double* x_covariates_pred, const double* theta6,
                        const double* smooth_limits, double* out);

/* Replaces `_cocons_cov_rns_classic` (src/RcppExports.cpp:59-69 -> cov_rns_classic,
 * src/cocons_full.cpp:480-594).  out: n x n. */
int cocons_cov_rns_classic(int64_t n, int64_t p, const double* locs, const double* x_covariates,
                           const double* theta6, double* out);

/* Replaces `_cocons_sumsmoothlone` (src/RcppExports.cpp:16-26 -> sumsmoothlone,
 * src/cocons_full.cpp:12-30).  A p-length host reduction; stays on the host. */
double cocons_sumsmoothlone(const double* x, int64_t len, double lambda, double alpha);

/* qr(X)$rank as base R computes it (LINPACK dqrdc2 with limited column pivoting, tol = 1e-7), which
 * GetNeg2loglikelihoodREML evaluates at R/neg2loglikelihood.R:270.  X is n x p column-major.  Host code. */
int cocons_qr_rank(const double* x, int64_t n, int64_t p, double tol);

/* ---- likelihood context: theta-independent inputs resident on the device -
 *
 * One context per (device, data set).  locs n x 2, x_covariates n x p, z n x r
 * are uploaded once; they are constant over the thousands of objective calls
 * of one cocoOptim run (R/optim.R:237-251).  `stream` is a cudaStream_t to
 * launch on (NULL: the context creates its own).  Sites are re-ordered along
 * a Morton curve inside the context (the likelihood is invariant to it). */
int cocons_ctx_create(int device, int64_t n, int64_t p, int64_t r, const double* locs, const double* x_covariates,
                      const double* z, void* stream, cocons_ctx** out);
void cocons_ctx_destroy(cocons_ctx* ctx);
/* dims4 = {n, p, r, q} of the resident data (q = 0 until cocons_ctx_set_xbetas); lets the .Call glue refuse
 * arguments whose shapes do not match the context before any pointer is handed to the device */
int cocons_ctx_dims(cocons_ctx* ctx, int64_t* dims4);

/* replace z (n x r, same r) - e.g. the REML contrasts of R/optim.R:311 */
int cocons_ctx_set_z(cocons_ctx* ctx, const double* z);
/* mean design for COCONS_PROFILE: x_betas n x q (R/optim.R:281) */
int cocons_ctx_set_xbetas(cocons_ctx* ctx, int64_t q, const double* x_betas);

/* One objective evaluation: assembly (lower triangle, in place) -> blocked
 * Cholesky -> log-determinant + forward solves + Gram reductions.
 *
 *   mean_p : p mean coefficients (ML: trend = X mean, R/neg2loglikelihood.R:210);
 *            may be NULL for PROFILE/REML.
 * Outputs (host):
 *   logdet     sum(log(diag(chol(Sigma))))            (:208)
 *   quad[r]    per column of z: ML  |R^-T (z - X mean)|^2  (:214-217)
 *                               PROFILE/REML  z' P z       (:157, :285)
 *   logdet_w   sum(log(diag(chol(W)))), W = X' Sigma^-1 X  (REML :280-285; 0 for ML)
 *   rank_x     qr(X)$rank as used at :270 (REML; 0 otherwise)
 * The caller adds n log(2 pi), the penalty and the `safe` logic, which stay
 * the reference's own host code.  Returns k > 0 when Sigma is not PD. */
int cocons_n2ll(cocons_ctx* ctx, int kind, const double* theta6, const double* smooth_limits, const double* mean_p,
                double* logdet, double* quad, double* logdet_w, int* rank_x);

/* ---- sparse (tapered) model, src/cocons_taper.cpp ------------------------
 * The pattern is spam's CSR layout as the reference receives it: 1-based
 * `colindices` (nnz) and `rowpointers` (rows + 1), INTSXP slots of the spam
 * object (Rcpp coerces them to doubles for the reference; here they stay
 * 32-bit integers). */

/* Replaces `_cocons_cov_rns_taper` (src/RcppExports.cpp:90-104 -> cov_rns_taper,
 * src/cocons_taper.cpp:151-433).  out: nnz covariance entries in pattern order
 * (the caller multiplies them into the taper, R/neg2loglikelihood.R:26). */
int cocons_cov_rns_taper(int64_t n, int64_t p, const double* locs, const double* x_covariates, const double* theta6,
                         const double* smooth_limits, const int32_t* colindices, const int32_t* rowpointers,
                         int64_t nnz, double* out);

/* Replaces `_cocons_cov_rns_taper_pred` (src/RcppExports.cpp:71-88 -> cov_rns_taper_pred,
 * src/cocons_taper.cpp:17-139).  The pattern has m rows (prediction sites) and n columns. */
int cocons_cov_rns_taper_pred(int64_t n, int64_t m, int64_t p, const double* locs, const double* locs_pred,
                              const double* x_covariates, const double* x_covariates_pred, const double* theta6,
                              const double* smooth_limits, const int32_t* colindices, const int32_t* rowpointers,
                              int64_t nnz, double* out);

/* Attach the taper of a sparse coco object to a context: the pattern of
 * `ref_taper` (n x n, caller order) and its entries (R/optim.R:376-379). */
int cocons_ctx_set_taper(cocons_ctx* ctx, const int32_t* colindices, const int32_t* rowpointers,
                         const double* taper_entries, int64_t nnz);

/* A context for the tapered model only, with the pattern fixed at creation: only the tiles of L that can be nonzero
 * (pattern + fill, Morton order) are stored, so n is bounded by the factor's fill, not by n_pad^2.  The pattern and
 * taper entries are those of cocons_ctx_set_taper; 0 <= r <= 128.  On such a context cocons_n2ll_taper,
 * cocons_factor_taper, cocons_ctx_get_factor (dense expansion, for small n), cocons_ctx_factor_rows,
 * cocons_ctx_set_z, cocons_ctx_dims, cocons_ctx_timings and cocons_ctx_destroy work as on a dense context; every
 * other context entry returns COCONS_ERR_STATE.  The factor differs from the dense path's in the last bits only. */
int cocons_ctx_create_taper_tiled(int device, int64_t n, int64_t p, int64_t r, const double* locs,
                                  const double* x_covariates, const double* z, const int32_t* colindices,
                                  const int32_t* rowpointers, const double* taper_entries, int64_t nnz,
                                  void* stream, cocons_ctx** out);
/* {tile columns, stored tiles, stored tiles outside the pattern (fill), tile products per factorisation} of a tiled
 * context: lower 128 x 128 tiles, diagonal included; a tile product is one 128 x 128 x 128 block of the trailing
 * updates (sum over tile columns of m (m + 1) / 2, m = stored tiles below the diagonal).  COCONS_ERR_STATE on a dense
 * context. */
int cocons_ctx_tile_stats(cocons_ctx* ctx, int64_t* stats4);

/* GetNeg2loglikelihoodTaper / ...TaperProfile (R/neg2loglikelihood.R:20-108):
 * taper * cov_rns_taper on the pattern -> Cholesky -> log-determinant and
 * |R^-T (z - X mean)|^2 per column of z.  Where the reference updates spam's
 * sparse Cholesky, the product is scattered into the dense lower triangle and
 * factored by the same blocked DMMA Cholesky (determinant and quadratic form
 * do not depend on spam's fill-reducing permutation).  The caller composes
 * the value (the Profile variant sets std.dev[1] = 0 before the call, :78). */
int cocons_n2ll_taper(cocons_ctx* ctx, const double* theta6, const double* smooth_limits, const double* mean_p,
                      double* logdet, double* quad);

/* Assemble taper * cov_rns_taper and factor it, keeping L on the device
 * (cocoPredict / cocoSim / getCovMatrix sparse branches, R/predict.R:219-231, R/sim.R:193-204). */
int cocons_factor_taper(cocons_ctx* ctx, const double* theta6, const double* smooth_limits);

/* cocoPredict sparse branch (R/predict.R:233-275) on the factor kept by
 * cocons_factor_taper.  The pattern (m rows x n columns) and `taper_entries`
 * are those of `pred_taper` before its entries are multiplied by
 * cov_rns_taper_pred - that product is formed on the device.  Outputs as
 * cocons_predict: stochastic = resid' Sigma^-1 C' (:259),
 * explained = rowSums(C * t(Sigma^-1 C')) (:274; NULL to skip). */
int cocons_predict_taper(cocons_ctx* ctx, int64_t m, const double* locs_pred, const double* x_covariates_pred,
                         const int32_t* colindices, const int32_t* rowpointers, const double* taper_entries,
                         int64_t nnz, const double* resid, double* stochastic, double* explained);

/* Profiled mean coefficients after a pml/reml fit (R/optim.R:326-343):
 * betas[q] = W^-1 V' rowSums(z) / r for the factor of the last cocons_n2ll /
 * cocons_factor call.  kind selects x_betas (PROFILE) or the full design (REML). */
int cocons_profile_betas(cocons_ctx* ctx, int kind, double* betas);

/* Assemble + factor only, keeping L on the device for predict / simulate.
 * par: COCONS_PAR_DIFF or COCONS_PAR_CLASSIC. */
int cocons_factor(cocons_ctx* ctx, int par, const double* theta6, const double* smooth_limits);

/* cocoPredict dense branch (R/predict.R:136-187) on the kept factor.
 * resid = z[,index] - X mean (n, host).  Outputs (m each, host):
 *   stochastic = resid' Sigma^-1 C'        (:150-159)
 *   explained  = rowSums(C * t(Sigma^-1 C'))  (:173)  (NULL to skip)
 * The caller forms sd.pred from `explained` as at :170-183. */
int cocons_predict(cocons_ctx* ctx, int64_t m, const double* locs_pred, const double* x_covariates_pred,
                   const double* resid, double* stochastic, double* explained);

/* cocoSim marginal branch (R/sim.R:162-172): out (n x k) = t(t(eps) %*% chol(Sigma)),
 * i.e. L eps, eps n x k standard normal draws made by the caller (R's RNG). */
int cocons_sim(cocons_ctx* ctx, int64_t k, const double* eps, double* out);

/* cocoSim conditional branch (R/sim.R:87-121): Schur complement of the
 * prediction sites given the kept factor, its Cholesky factor applied to eps
 * (m x k).  out (m x k) = t(t(eps) %*% chol(S_pp - S_po S_oo^-1 S_op)). */
int cocons_sim_cond(cocons_ctx* ctx, int64_t m, const double* locs_pred, const double* x_covariates_pred,
                    int64_t k, const double* eps, double* out);

/* Copy the kept factor (lower triangle, n x n, zeros above) back in the
 * caller's original site order is not possible after Morton re-ordering, so
 * this returns L of the re-ordered matrix together with the permutation
 * (perm[i] = original index of re-ordered site i).  For tests. */
int cocons_ctx_get_factor(cocons_ctx* ctx, double* L, int64_t* perm);

/* Rows of the kept factor for m caller-order sites: rows[a*n + k] = L[pos[a], k] (zero for k > pos[a]),
 * pos[a] = position of sites[a] in the re-ordered matrix.  (L L^T)[pos[a], pos[b]] is then the covariance of
 * sites a and b (base::chol, R/neg2loglikelihood.R:200): the residual check of the factorisation at sizes
 * whose full factor does not fit a host (n = 100 000: 80 GB). */
int cocons_ctx_factor_rows(cocons_ctx* ctx, const int64_t* sites, int64_t m, double* rows, int64_t* pos);

/* Host only, for tests: the work units of the forward substitution (csrc/solve.cu, K6b) for an n_pad x n_pad factor, in
 * issue order, 4 ints each (tile row, first tile column, end tile column, chunk).  Returns their number (units4 may be
 * NULL); no device is touched.  (forwardsolve, R/neg2loglikelihood.R:214-217) */
int64_t cocons_debug_solve_units(int64_t n_pad, int32_t* units4, int64_t capacity);

/* per-phase device times of the last evaluation, milliseconds (CUDA events on
 * the context's stream): [0] site+assembly [1] factorisation [2] solves+reductions [3] total */
int cocons_ctx_timings(cocons_ctx* ctx, double* ms4);

/* debugging aid: with COCONS_DEBUG_CHECKSUM=1 in the environment every evaluation also forms the
 * (deterministic) sum of the lower triangle after the assembly [0] and after the factorisation [1];
 * used by tools/pool_stress.py to localise differences between concurrent evaluations */
int cocons_ctx_debug_checksums(cocons_ctx* ctx, double* out2);

/* duration (ms, CUDA events inside the evaluation) and flop count of the LARGEST trailing-update launch of
 * the last factorisation - the dominant kernel's own roofline point (bench.py) */
int cocons_ctx_kernel_timing(cocons_ctx* ctx, double* ms, double* flops);

/* ---- one-shot objective, host buffers in, scalars out ------------------
 * What the R closure GetNeg2loglikelihood{,Profile,REML} binds to: uploads
 * locs / X / z / x_betas every call (they arrive as R objects every call),
 * reuses a per-process workspace keyed on (device, n, p, r, q). */
int cocons_neg2loglik_dense(int kind, int64_t n, int64_t p, int64_t r, int64_t q, const double* locs,
                            const double* x_covariates, const double* z, const double* x_betas,
                            const double* theta6, const double* smooth_limits, const double* mean_p, double* logdet,
                            double* quad, double* logdet_w, int* rank_x);
/* release the per-process workspace of cocons_neg2loglik_dense */
void cocons_release_workspace(void);

/* ---- multi-GPU: one rank's half of the block-cyclic factorisation ------------------------
 * For matrices beyond one GPU (n = 200 000).  One process per GPU; column panels of 512 are
 * dealt round-robin to the ranks.  The exchange step (broadcast of a packed panel, small
 * reductions in the solve) is issued by the host driver over NCCL on device buffers IT owns
 * (cocons_b200/distributed.py; an R host would use the same calls from one worker per GPU).
 * All `void*` arguments below are device pointers. */
typedef struct cocons_dist cocons_dist;
int cocons_dist_create(int device, int rank, int world, int64_t n, int64_t p, int64_t r, const double* locs,
                       const double* x_covariates, const double* z, void* stream, cocons_dist** out);
void cocons_dist_destroy(cocons_dist* ctx);
int cocons_dist_set_xbetas(cocons_dist* ctx, int64_t q, const double* x_betas);
int64_t cocons_dist_npanels(cocons_dist* ctx);
int64_t cocons_dist_npad(cocons_dist* ctx);
int64_t cocons_dist_panel_elems(cocons_dist* ctx, int64_t K);
int cocons_dist_assemble(cocons_dist* ctx, const double* theta6, const double* smooth_limits, const double* mean_p);
void* cocons_dist_side_stream(cocons_dist* ctx);
int cocons_dist_factor_panel(cocons_dist* ctx, int64_t K, int side);
int cocons_dist_pack_panel(cocons_dist* ctx, int64_t K, void* dst, int side);
int cocons_dist_update(cocons_dist* ctx, int64_t K, const void* src, int64_t J_lo, int64_t J_hi);
int cocons_dist_fill_rhs(cocons_dist* ctx, int kind, void* rhs, int* nr_out);
int cocons_dist_solve_block(cocons_dist* ctx, int64_t K, const void* bK, const void* tK, void* acc, void* Y, int nr);
int cocons_dist_reduce_local(cocons_dist* ctx, const void* Y, int nr, void* out2, void* gram);
int cocons_dist_perm(cocons_dist* ctx, int64_t* perm);

/* ---- measurement helpers (bench.py) -------------------------------------
 * C (n x n, device-resident inside the call) -= A A' with the DMMA trailing-
 * update kernel, timed with CUDA events; returns milliseconds per repetition.
 * Used to report the kernel's standalone FP64 rate next to cuBLAS dgemm. */
int cocons_bench_syrk(int device, int64_t n, int64_t k, int reps, double* ms_per_rep);
/* The K = 768 trailing update of the factorisation, C (m x m) -= P P' over the
 * lower 128 x 64 tiles, with P m x 768, both column-major, m a multiple of 128.
 * path 0: the DMMA kernel; 1: the split-int8 kernel (split of P included;
 * COCONS_ERR_STATE if the library was built without it).  P and C given: C is
 * updated once in place.  Both null: constant device data.  reps > 0: that
 * many further updates are timed with CUDA events (ms per repetition). */
int cocons_trailing_update(int device, int64_t m, const double* P, double* C, int path, int reps,
                           double* ms_per_rep);

#ifdef __cplusplus
}
#endif

#endif /* COCONS_B200_H */
