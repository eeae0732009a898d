/* .Call glue between the R package and libcocons_b200 - the hand-written replacement for the
 * Rcpp-generated src/RcppExports.cpp of the reference (its wrappers :16-103, the registration
 * table :105-113 and R_init_cocons :115-118).  Plain C on R's C API, no Rcpp.
 *
 * Build inside the R package:  R CMD SHLIB cocons_glue.c -L<dir> -lcocons_b200 -o cocons.so
 * (see INTEGRATION.md).  R is not available in the build image of this repository, so here the
 * file is compiled against the declarations in rglue/stub/ and EXECUTED against a miniature of R's
 * C API (tests/rmock: garbage collection at every allocation, PROTECT-stack and malloc accounting,
 * Rf_error unwinding) by tests/test_rglue.py - on the CPU for registration, argument handling and
 * error paths, on the GPU (-m gpu) for the same .Call sequences an R session makes, against the goldens.
 *
 * Every argument check that can raise an R error runs before anything is malloc'd (Rf_error does
 * not return), and every shape is checked before a pointer is handed to the library: the
 * reference's Rcpp code reads matrices through unchecked operator(), a mismatch here would make
 * the device read past a host buffer.
 *
 * Conventions kept from the reference:
 *   - `theta` is a named list; aspects are looked up BY NAME ("std.dev","scale","aniso","tilt",
 *     "smooth","nugget", src/cocons_full.cpp:47-54), extra names such as "mean" are ignored and
 *     a missing name is an error;
 *   - integer matrices / vectors are silently coerced to double, as Rcpp's input_parameter<> does
 *     (src/RcppExports.cpp:34-36);
 *   - results are freshly allocated REALSXP matrices with a `dim` attribute and no dimnames;
 *     inputs are never written to.
 * Errors: a negative status from the library becomes an R error (raised after every temporary
 * has been released); a positive status (matrix not positive definite) is handed back to the R
 * caller, which applies the reference's own `safe` / 1e6 logic (R/neg2loglikelihood.R:200-206).
 * CUDA is initialised lazily on the first call in each process, never at load time, so forked
 * optimParallel workers (R/optim.R:117-121) each get their own context.
 */
#include <R.h>
#include <Rinternals.h>
#include <R_ext/Rdynload.h>

#include "../../include/cocons_b200.h"

static const char* const kAspects[6] = {"std.dev", "scale", "aniso", "tilt", "smooth", "nugget"};

/* coerce to REALSXP (caller PROTECTs) */
static SEXP as_real(SEXP x) { return TYPEOF(x) == REALSXP ? x : Rf_coerceVector(x, REALSXP); }

static SEXP list_get(SEXP list, const char* name) {
  SEXP names = Rf_getAttrib(list, R_NamesSymbol);
  if (TYPEOF(list) != VECSXP || Rf_isNull(names)) Rf_error("theta must be a named list");
  for (R_xlen_t i = 0; i < XLENGTH(list); ++i)
    if (strcmp(CHAR(STRING_ELT(names, i)), name) == 0) return VECTOR_ELT(list, i);
  Rf_error("Index out of bounds: [index='%s'].", name);
}

/* named list -> 6 x p block (malloc'd; caller frees), all aspects must have length p.  Every check that can raise
 * an R error runs BEFORE the buffer exists: Rf_error() does not return, so nothing may be owned when it is called */
static double* pack_theta(SEXP theta, int p) {
  SEXP part[6];
  for (int a = 0; a < 6; ++a) {
    part[a] = PROTECT(as_real(list_get(theta, kAspects[a])));
    if (LENGTH(part[a]) != p) Rf_error("theta$%s has length %d, expected %d", kAspects[a], LENGTH(part[a]), p);
  }
  double* out = (double*)malloc(sizeof(double) * 6 * (size_t)(p > 0 ? p : 1));
  if (!out) Rf_error("out of memory");
  for (int a = 0; a < 6; ++a) memcpy(out + (size_t)a * p, REAL(part[a]), sizeof(double) * (size_t)p);
  UNPROTECT(6);
  return out;
}

/* shape checks the reference leaves to Rcpp's bounds-unchecked operator(): here a mismatch would make the device
 * read past a host buffer, so it is an R error instead */
static void need(int ok, const char* who, const char* what) {
  if (!ok) Rf_error("%s: %s", who, what);
}
static int rows_of(SEXP x) { return Rf_isMatrix(x) ? Rf_nrows(x) : LENGTH(x); }
static void check_sites(const char* who, SEXP locs, SEXP x) {
  need(Rf_isMatrix(locs) && Rf_ncols(locs) == 2, who, "locs must be a matrix with two columns");
  need(Rf_isMatrix(x) && Rf_nrows(x) == Rf_nrows(locs), who, "x_covariates must be a matrix with nrow(locs) rows");
  need(Rf_nrows(locs) >= 1 && Rf_ncols(x) >= 1, who, "empty design");
}
static void check_limits(const char* who, SEXP lim) {
  need(LENGTH(lim) == 2, who, "smooth_limits must have two elements");
}

static void raise(int status) {
  if (status < 0) Rf_error("cocons_b200: %s", cocons_last_error());
}

/* ---- the reference's six registered entry points -------------------------------------- */

SEXP _cocons_sumsmoothlone(SEXP xS, SEXP lambdaS, SEXP alphaS) {
  SEXP x = PROTECT(as_real(xS));
  double v = cocons_sumsmoothlone(REAL(x), XLENGTH(x), Rf_asReal(lambdaS), Rf_asReal(alphaS));
  UNPROTECT(1);
  return Rf_ScalarReal(v);
}

SEXP _cocons_cov_rns(SEXP thetaS, SEXP locsS, SEXP xS, SEXP limS) {
  SEXP locs = PROTECT(as_real(locsS)), x = PROTECT(as_real(xS)), lim = PROTECT(as_real(limS));
  check_sites("cov_rns", locs, x);
  check_limits("cov_rns", lim);
  const int n = Rf_nrows(locs), p = Rf_ncols(x);
  double* th = pack_theta(thetaS, p);
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, n, n));
  int rc = cocons_cov_rns(n, p, REAL(locs), REAL(x), th, REAL(lim), REAL(out));
  free(th);
  UNPROTECT(4);
  raise(rc);
  return out;
}

SEXP _cocons_cov_rns_pred(SEXP thetaS, SEXP locsS, SEXP locsPredS, SEXP xS, SEXP xPredS, SEXP limS) {
  SEXP locs = PROTECT(as_real(locsS)), lp = PROTECT(as_real(locsPredS));
  SEXP x = PROTECT(as_real(xS)), xp = PROTECT(as_real(xPredS)), lim = PROTECT(as_real(limS));
  check_sites("cov_rns_pred", locs, x);
  check_sites("cov_rns_pred", lp, xp);
  need(Rf_ncols(xp) == Rf_ncols(x), "cov_rns_pred", "x_covariates_pred and x_covariates differ in columns");
  check_limits("cov_rns_pred", lim);
  const int n = Rf_nrows(locs), m = Rf_nrows(lp), p = Rf_ncols(x);
  double* th = pack_theta(thetaS, p);
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, m, n));
  int rc = cocons_cov_rns_pred(n, m, p, REAL(locs), REAL(lp), REAL(x), REAL(xp), th, REAL(lim), REAL(out));
  free(th);
  UNPROTECT(6);
  raise(rc);
  return out;
}

SEXP _cocons_cov_rns_classic(SEXP thetaS, SEXP locsS, SEXP xS) {
  SEXP locs = PROTECT(as_real(locsS)), x = PROTECT(as_real(xS));
  check_sites("cov_rns_classic", locs, x);
  const int n = Rf_nrows(locs), p = Rf_ncols(x);
  double* th = pack_theta(thetaS, p);
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, n, n));
  int rc = cocons_cov_rns_classic(n, p, REAL(locs), REAL(x), th, REAL(out));
  free(th);
  UNPROTECT(3);
  raise(rc);
  return out;
}

/* spam's colindices / rowpointers slots are INTSXP; the reference's Rcpp wrappers accept any numeric
 * vector for them (src/RcppExports.cpp:81-82, 99-100), so doubles are coerced too */
static SEXP as_int(SEXP x) { return TYPEOF(x) == INTSXP ? x : Rf_coerceVector(x, INTSXP); }

SEXP _cocons_cov_rns_taper_pred(SEXP thetaS, SEXP locsS, SEXP locsPredS, SEXP xS, SEXP xPredS, SEXP colS, SEXP rowS,
                                SEXP limS) {
  SEXP locs = PROTECT(as_real(locsS)), lp = PROTECT(as_real(locsPredS));
  SEXP x = PROTECT(as_real(xS)), xp = PROTECT(as_real(xPredS)), lim = PROTECT(as_real(limS));
  SEXP col = PROTECT(as_int(colS)), row = PROTECT(as_int(rowS));
  check_sites("cov_rns_taper_pred", locs, x);
  check_sites("cov_rns_taper_pred", lp, xp);
  need(Rf_ncols(xp) == Rf_ncols(x), "cov_rns_taper_pred", "x_covariates_pred and x_covariates differ in columns");
  check_limits("cov_rns_taper_pred", lim);
  const int n = Rf_nrows(locs), m = Rf_nrows(lp), p = Rf_ncols(x);
  need(LENGTH(row) == m + 1, "cov_rns_taper_pred", "rowpointers must have nrow(locs_pred) + 1 elements");
  double* th = pack_theta(thetaS, p);
  SEXP out = PROTECT(Rf_allocVector(REALSXP, XLENGTH(col)));
  int rc = cocons_cov_rns_taper_pred(n, m, p, REAL(locs), REAL(lp), REAL(x), REAL(xp), th, REAL(lim), INTEGER(col),
                                     INTEGER(row), XLENGTH(col), REAL(out));
  free(th);
  UNPROTECT(8);
  raise(rc);
  return out;
}

SEXP _cocons_cov_rns_taper(SEXP thetaS, SEXP locsS, SEXP xS, SEXP colS, SEXP rowS, SEXP limS) {
  SEXP locs = PROTECT(as_real(locsS)), x = PROTECT(as_real(xS)), lim = PROTECT(as_real(limS));
  SEXP col = PROTECT(as_int(colS)), row = PROTECT(as_int(rowS));
  check_sites("cov_rns_taper", locs, x);
  check_limits("cov_rns_taper", lim);
  const int n = Rf_nrows(locs), p = Rf_ncols(x);
  need(LENGTH(row) == n + 1, "cov_rns_taper", "rowpointers must have nrow(locs) + 1 elements");
  double* th = pack_theta(thetaS, p);
  SEXP out = PROTECT(Rf_allocVector(REALSXP, XLENGTH(col)));
  int rc = cocons_cov_rns_taper(n, p, REAL(locs), REAL(x), th, REAL(lim), INTEGER(col), INTEGER(row), XLENGTH(col),
                                REAL(out));
  free(th);
  UNPROTECT(6);
  raise(rc);
  return out;
}

/* ---- fused objective: what GetNeg2loglikelihood{,Profile,REML} call --------------------- */

/* returns c(status, logdet, logdet_w, rank, quad_1..quad_r) */
SEXP _cocons_n2ll_dense(SEXP kindS, SEXP thetaS, SEXP locsS, SEXP xS, SEXP limS, SEXP zS, SEXP xbS, SEXP meanS) {
  SEXP locs = PROTECT(as_real(locsS)), x = PROTECT(as_real(xS)), lim = PROTECT(as_real(limS));
  SEXP z = PROTECT(as_real(zS)), mean = PROTECT(as_real(meanS));
  SEXP xb = PROTECT(Rf_isNull(xbS) ? xbS : as_real(xbS));
  check_sites("n2ll_dense", locs, x);
  check_limits("n2ll_dense", lim);
  const int n = Rf_nrows(locs), p = Rf_ncols(x);
  const int r = Rf_isMatrix(z) ? Rf_ncols(z) : 1;
  const int q = Rf_isNull(xb) ? 0 : (Rf_isMatrix(xb) ? Rf_ncols(xb) : 1);
  need(rows_of(z) == n, "n2ll_dense", "z must have nrow(locs) rows");
  need(q == 0 || rows_of(xb) == n, "n2ll_dense", "x_betas must have nrow(locs) rows");
  double* th = pack_theta(thetaS, p);
  SEXP out = PROTECT(Rf_allocVector(REALSXP, 4 + r));
  double logdet = R_NaReal, ldw = 0.0;
  int rank = 0;
  int rc = cocons_neg2loglik_dense(Rf_asInteger(kindS), n, p, r, q, REAL(locs), REAL(x), REAL(z),
                                   q ? REAL(xb) : NULL, th, REAL(lim), LENGTH(mean) == p ? REAL(mean) : NULL, &logdet,
                                   REAL(out) + 4, &ldw, &rank);
  free(th);
  REAL(out)[0] = rc, REAL(out)[1] = logdet, REAL(out)[2] = ldw, REAL(out)[3] = rank;
  UNPROTECT(7);
  raise(rc);
  return out;
}

/* ---- device-resident context behind an external pointer --------------------------------- */

static void ctx_finalizer(SEXP ptr) {
  if (TYPEOF(ptr) != EXTPTRSXP) return;
  cocons_ctx* c = (cocons_ctx*)R_ExternalPtrAddr(ptr);
  if (c) cocons_ctx_destroy(c);
  R_ClearExternalPtr(ptr);
}

static cocons_ctx* ctx_of(SEXP ptr) {
  if (TYPEOF(ptr) != EXTPTRSXP) Rf_error("cocons_b200: not a context (external pointer expected)");
  cocons_ctx* c = (cocons_ctx*)R_ExternalPtrAddr(ptr);
  if (!c) Rf_error("cocons_b200: the context has been released");
  return c;
}

SEXP _cocons_ctx_new(SEXP locsS, SEXP xS, SEXP zS, SEXP deviceS) {
  SEXP locs = PROTECT(as_real(locsS)), x = PROTECT(as_real(xS)), z = PROTECT(as_real(zS));
  check_sites("ctx_new", locs, x);
  need(rows_of(z) == Rf_nrows(locs), "ctx_new", "z must have nrow(locs) rows");
  const int n = Rf_nrows(locs), p = Rf_ncols(x), r = Rf_isMatrix(z) ? Rf_ncols(z) : 1;
  cocons_ctx* c = NULL;
  int rc = cocons_ctx_create(Rf_asInteger(deviceS), n, p, r, REAL(locs), REAL(x), REAL(z), NULL, &c);
  UNPROTECT(3);
  raise(rc);
  SEXP ptr = PROTECT(R_MakeExternalPtr(c, R_NilValue, R_NilValue));
  R_RegisterCFinalizerEx(ptr, ctx_finalizer, TRUE);
  UNPROTECT(1);
  return ptr;
}

SEXP _cocons_ctx_free(SEXP ptr) {
  ctx_finalizer(ptr);
  return R_NilValue;
}

/* {n, p, r, q} of a live context */
typedef struct {
  cocons_ctx* c;
  int n, p, r, q;
} ctx_view;

static ctx_view view_of(SEXP ptr) {
  ctx_view v;
  int64_t d[4] = {0, 0, 0, 0};
  v.c = ctx_of(ptr);
  if (cocons_ctx_dims(v.c, d) != 0) Rf_error("cocons_b200: %s", cocons_last_error());
  v.n = (int)d[0], v.p = (int)d[1], v.r = (int)d[2], v.q = (int)d[3];
  return v;
}

/* prediction sites against a context: m x 2 coordinates, m x p design */
static int check_pred_sites(const char* who, const ctx_view* v, SEXP lp, SEXP xp) {
  need(Rf_isMatrix(lp) && Rf_ncols(lp) == 2, who, "locs_pred must be a matrix with two columns");
  need(Rf_isMatrix(xp) && Rf_nrows(xp) == Rf_nrows(lp) && Rf_ncols(xp) == v->p, who,
       "x_covariates_pred must be nrow(locs_pred) x p");
  return Rf_nrows(lp);
}

SEXP _cocons_ctx_set_z(SEXP ptr, SEXP zS) {
  const ctx_view v = view_of(ptr);
  SEXP z = PROTECT(as_real(zS));
  need(XLENGTH(z) == (R_xlen_t)v.n * v.r, "ctx_set_z", "z must be n x r like the z the context was created with");
  int rc = cocons_ctx_set_z(v.c, REAL(z));
  UNPROTECT(1);
  raise(rc);
  return R_NilValue;
}

SEXP _cocons_ctx_set_xbetas(SEXP ptr, SEXP xbS) {
  const ctx_view v = view_of(ptr);
  SEXP xb = PROTECT(as_real(xbS));
  need(rows_of(xb) == v.n, "ctx_set_xbetas", "x_betas must have n rows");
  int rc = cocons_ctx_set_xbetas(v.c, Rf_isMatrix(xb) ? Rf_ncols(xb) : 1, REAL(xb));
  UNPROTECT(1);
  raise(rc);
  return R_NilValue;
}

/* c(status, logdet, logdet_w, rank, quad...) on the resident data */
SEXP _cocons_ctx_n2ll(SEXP ptr, SEXP kindS, SEXP thetaS, SEXP pS, SEXP rS, SEXP limS, SEXP meanS) {
  const ctx_view v = view_of(ptr);
  SEXP lim = PROTECT(as_real(limS)), mean = PROTECT(as_real(meanS));
  const int p = Rf_asInteger(pS), r = Rf_asInteger(rS);
  need(p == v.p && r == v.r, "ctx_n2ll", "p / r differ from the context's");
  check_limits("ctx_n2ll", lim);
  double* th = pack_theta(thetaS, p);
  SEXP out = PROTECT(Rf_allocVector(REALSXP, 4 + r));
  double logdet = R_NaReal, ldw = 0.0;
  int rank = 0;
  int rc = cocons_n2ll(v.c, Rf_asInteger(kindS), th, REAL(lim), LENGTH(mean) == p ? REAL(mean) : NULL, &logdet,
                       REAL(out) + 4, &ldw, &rank);
  free(th);
  REAL(out)[0] = rc, REAL(out)[1] = logdet, REAL(out)[2] = ldw, REAL(out)[3] = rank;
  UNPROTECT(3);
  raise(rc);
  return out;
}

/* ---- batch context: many points per call (cocons_ctx_create_batch) ------------------------------------------------ */

SEXP _cocons_ctx_new_batch(SEXP locsS, SEXP xS, SEXP zS, SEXP batchS, SEXP deviceS) {
  SEXP locs = PROTECT(as_real(locsS)), x = PROTECT(as_real(xS)), z = PROTECT(as_real(zS));
  check_sites("ctx_new_batch", locs, x);
  need(rows_of(z) == Rf_nrows(locs), "ctx_new_batch", "z must have nrow(locs) rows");
  const int batch = Rf_asInteger(batchS);
  need(batch >= 1, "ctx_new_batch", "batch must be a positive integer");
  const int n = Rf_nrows(locs), p = Rf_ncols(x), r = Rf_isMatrix(z) ? Rf_ncols(z) : 1;
  cocons_ctx* c = NULL;
  int rc = cocons_ctx_create_batch(Rf_asInteger(deviceS), n, p, r, REAL(locs), REAL(x), REAL(z), batch, NULL, &c);
  UNPROTECT(3);
  raise(rc);
  SEXP ptr = PROTECT(R_MakeExternalPtr(c, R_NilValue, R_NilValue));
  R_RegisterCFinalizerEx(ptr, ctx_finalizer, TRUE);
  UNPROTECT(1);
  return ptr;
}

/* list(logdet[npoints], quad (r x npoints), logdet_w[npoints], rank_x, status[npoints]) for a list of named theta
 * lists and a list of mean vectors (or NULL); status[i] is what _cocons_ctx_n2ll's status would be for point i */
SEXP _cocons_ctx_n2ll_batch(SEXP ptr, SEXP kindS, SEXP thetasS, SEXP pS, SEXP rS, SEXP limS, SEXP meansS) {
  const ctx_view v = view_of(ptr);
  SEXP lim = PROTECT(as_real(limS));
  const int p = Rf_asInteger(pS), r = Rf_asInteger(rS);
  need(p == v.p && r == v.r, "ctx_n2ll_batch", "p / r differ from the context's");
  check_limits("ctx_n2ll_batch", lim);
  need(TYPEOF(thetasS) == VECSXP && XLENGTH(thetasS) >= 1, "ctx_n2ll_batch", "thetas must be a non-empty list");
  const int npts = LENGTH(thetasS);
  need(Rf_isNull(meansS) || (TYPEOF(meansS) == VECSXP && LENGTH(meansS) == npts), "ctx_n2ll_batch",
       "means must be NULL or a list with one vector per point");
  /* every check that can raise an R error before the buffers exist (pack_theta raises only before its malloc) */
  for (int i = 0; i < npts; ++i) {
    free(pack_theta(VECTOR_ELT(thetasS, i), p));
    if (!Rf_isNull(meansS)) need(LENGTH(VECTOR_ELT(meansS, i)) == p, "ctx_n2ll_batch", "every mean must have length p");
  }
  SEXP means = PROTECT(Rf_allocVector(VECSXP, Rf_isNull(meansS) ? 0 : npts));
  for (int i = 0; !Rf_isNull(meansS) && i < npts; ++i) SET_VECTOR_ELT(means, i, as_real(VECTOR_ELT(meansS, i)));
  SEXP out = PROTECT(Rf_allocVector(VECSXP, 5));
  SEXP logdet = PROTECT(Rf_allocVector(REALSXP, npts)), quad = PROTECT(Rf_allocMatrix(REALSXP, r, npts));
  SEXP ldw = PROTECT(Rf_allocVector(REALSXP, npts)), status = PROTECT(Rf_allocVector(INTSXP, npts));
  for (int i = 0; i < npts; ++i) REAL(logdet)[i] = R_NaReal, REAL(ldw)[i] = 0.0;
  for (R_xlen_t i = 0; i < (R_xlen_t)r * npts; ++i) REAL(quad)[i] = R_NaReal;
  double* th = (double*)malloc(sizeof(double) * 6 * (size_t)p * npts);
  double* mean = Rf_isNull(meansS) ? NULL : (double*)malloc(sizeof(double) * (size_t)p * npts);
  const int oom = !th || (!mean && !Rf_isNull(meansS));
  int rc = 0, rank = 0;
  if (!oom) {
    for (int i = 0; i < npts; ++i) {
      double* one = pack_theta(VECTOR_ELT(thetasS, i), p);
      memcpy(th + (size_t)6 * p * i, one, sizeof(double) * 6 * (size_t)p);
      free(one);
      if (mean) memcpy(mean + (size_t)p * i, REAL(VECTOR_ELT(means, i)), sizeof(double) * (size_t)p);
    }
    rc = cocons_n2ll_batch(v.c, Rf_asInteger(kindS), npts, th, REAL(lim), mean, REAL(logdet), REAL(quad), REAL(ldw),
                           &rank, INTEGER(status));
  }
  free(th);
  free(mean);
  SET_VECTOR_ELT(out, 0, logdet);
  SET_VECTOR_ELT(out, 1, quad);
  SET_VECTOR_ELT(out, 2, ldw);
  SET_VECTOR_ELT(out, 3, Rf_ScalarInteger(rank));
  SET_VECTOR_ELT(out, 4, status);
  UNPROTECT(7);
  if (oom) Rf_error("out of memory");
  raise(rc);
  return out;
}

SEXP _cocons_ctx_factor(SEXP ptr, SEXP parS, SEXP thetaS, SEXP pS, SEXP limS) {
  const ctx_view v = view_of(ptr);
  SEXP lim = PROTECT(Rf_isNull(limS) ? limS : as_real(limS));
  need(Rf_asInteger(pS) == v.p, "ctx_factor", "p differs from the context's");
  if (!Rf_isNull(lim)) check_limits("ctx_factor", lim);
  double* th = pack_theta(thetaS, v.p);
  int rc = cocons_factor(v.c, Rf_asInteger(parS), th, Rf_isNull(lim) ? NULL : REAL(lim));
  free(th);
  UNPROTECT(1);
  raise(rc);
  return Rf_ScalarInteger(rc);
}

SEXP _cocons_ctx_profile_betas(SEXP ptr, SEXP kindS, SEXP qS) {
  const ctx_view v = view_of(ptr);
  const int kind = Rf_asInteger(kindS), q = Rf_asInteger(qS);
  need(q == (kind == COCONS_PROFILE ? v.q : v.p), "ctx_profile_betas", "q is not the number of mean columns");
  SEXP out = PROTECT(Rf_allocVector(REALSXP, q));
  int rc = cocons_profile_betas(v.c, kind, REAL(out));
  UNPROTECT(1);
  raise(rc);
  return out;
}

/* list(stochastic, explained) for cocoPredict (R/predict.R:150-173) */
SEXP _cocons_ctx_predict(SEXP ptr, SEXP locsPredS, SEXP xPredS, SEXP residS) {
  const ctx_view v = view_of(ptr);
  SEXP lp = PROTECT(as_real(locsPredS)), xp = PROTECT(as_real(xPredS)), resid = PROTECT(as_real(residS));
  const int m = check_pred_sites("ctx_predict", &v, lp, xp);
  need(XLENGTH(resid) == v.n, "ctx_predict", "the residual must have n elements");
  SEXP out = PROTECT(Rf_allocVector(VECSXP, 2));
  SEXP sto = PROTECT(Rf_allocVector(REALSXP, m)), expl = PROTECT(Rf_allocVector(REALSXP, m));
  int rc = cocons_predict(v.c, m, REAL(lp), REAL(xp), REAL(resid), REAL(sto), REAL(expl));
  SET_VECTOR_ELT(out, 0, sto);
  SET_VECTOR_ELT(out, 1, expl);
  UNPROTECT(6);
  raise(rc);
  return out;
}

/* ---- sparse (tapered) model on a resident context ----------------------------------------- */

/* attach ref_taper (its colindices / rowpointers / entries slots, R/optim.R:376-379) */
SEXP _cocons_ctx_set_taper(SEXP ptr, SEXP colS, SEXP rowS, SEXP entriesS) {
  const ctx_view v = view_of(ptr);
  SEXP col = PROTECT(as_int(colS)), row = PROTECT(as_int(rowS)), ent = PROTECT(as_real(entriesS));
  need(XLENGTH(ent) == XLENGTH(col), "ctx_set_taper", "entries and colindices differ in length");
  need(LENGTH(row) == v.n + 1, "ctx_set_taper", "rowpointers must have n + 1 elements");
  int rc = cocons_ctx_set_taper(v.c, INTEGER(col), INTEGER(row), REAL(ent), XLENGTH(col));
  UNPROTECT(3);
  raise(rc);
  return R_NilValue;
}

/* a context for the tapered model only, with ref_taper's pattern fixed: only the tiles of the Cholesky factor that can
 * be nonzero are stored (cocons_ctx_create_taper_tiled).  Same external-pointer class as _cocons_ctx_new, so
 * _cocons_ctx_n2ll_taper / _cocons_ctx_factor_taper / _cocons_ctx_set_z / _cocons_ctx_free take it as they are */
SEXP _cocons_ctx_new_taper_tiled(SEXP locsS, SEXP xS, SEXP zS, SEXP colS, SEXP rowS, SEXP entriesS, SEXP deviceS) {
  SEXP locs = PROTECT(as_real(locsS)), x = PROTECT(as_real(xS)), z = PROTECT(as_real(zS));
  SEXP col = PROTECT(as_int(colS)), row = PROTECT(as_int(rowS)), ent = PROTECT(as_real(entriesS));
  check_sites("ctx_new_taper_tiled", locs, x);
  need(rows_of(z) == Rf_nrows(locs), "ctx_new_taper_tiled", "z must have nrow(locs) rows");
  const int n = Rf_nrows(locs), p = Rf_ncols(x), r = Rf_isMatrix(z) ? Rf_ncols(z) : 1;
  need(r <= 128, "ctx_new_taper_tiled", "z may have at most 128 columns");
  need(XLENGTH(ent) == XLENGTH(col), "ctx_new_taper_tiled", "entries and colindices differ in length");
  need(LENGTH(row) == n + 1, "ctx_new_taper_tiled", "rowpointers must have nrow(locs) + 1 elements");
  cocons_ctx* c = NULL;
  int rc = cocons_ctx_create_taper_tiled(Rf_asInteger(deviceS), n, p, r, REAL(locs), REAL(x), REAL(z), INTEGER(col),
                                         INTEGER(row), REAL(ent), XLENGTH(col), NULL, &c);
  UNPROTECT(6);
  raise(rc);
  SEXP ptr = PROTECT(R_MakeExternalPtr(c, R_NilValue, R_NilValue));
  R_RegisterCFinalizerEx(ptr, ctx_finalizer, TRUE);
  UNPROTECT(1);
  return ptr;
}

/* c(status, logdet, quad...) of the tapered model (R/neg2loglikelihood.R:20-108) */
SEXP _cocons_ctx_n2ll_taper(SEXP ptr, SEXP thetaS, SEXP pS, SEXP rS, SEXP limS, SEXP meanS) {
  const ctx_view v = view_of(ptr);
  SEXP lim = PROTECT(as_real(limS)), mean = PROTECT(as_real(meanS));
  const int p = Rf_asInteger(pS), r = Rf_asInteger(rS);
  need(p == v.p && r == v.r, "ctx_n2ll_taper", "p / r differ from the context's");
  check_limits("ctx_n2ll_taper", lim);
  double* th = pack_theta(thetaS, p);
  SEXP out = PROTECT(Rf_allocVector(REALSXP, 2 + r));
  double logdet = R_NaReal;
  int rc = cocons_n2ll_taper(v.c, th, REAL(lim), LENGTH(mean) == p ? REAL(mean) : NULL, &logdet, REAL(out) + 2);
  free(th);
  REAL(out)[0] = rc, REAL(out)[1] = logdet;
  UNPROTECT(3);
  raise(rc);
  return out;
}

SEXP _cocons_ctx_factor_taper(SEXP ptr, SEXP thetaS, SEXP pS, SEXP limS) {
  const ctx_view v = view_of(ptr);
  SEXP lim = PROTECT(as_real(limS));
  need(Rf_asInteger(pS) == v.p, "ctx_factor_taper", "p differs from the context's");
  check_limits("ctx_factor_taper", lim);
  double* th = pack_theta(thetaS, v.p);
  int rc = cocons_factor_taper(v.c, th, REAL(lim));
  free(th);
  UNPROTECT(1);
  raise(rc);
  return Rf_ScalarInteger(rc);
}

/* list(stochastic, explained) for the sparse cocoPredict (R/predict.R:233-275); the pattern and entries are
 * those of pred_taper BEFORE the covariance is multiplied in */
SEXP _cocons_ctx_predict_taper(SEXP ptr, SEXP locsPredS, SEXP xPredS, SEXP colS, SEXP rowS, SEXP entriesS,
                               SEXP residS) {
  const ctx_view v = view_of(ptr);
  SEXP lp = PROTECT(as_real(locsPredS)), xp = PROTECT(as_real(xPredS)), resid = PROTECT(as_real(residS));
  SEXP col = PROTECT(as_int(colS)), row = PROTECT(as_int(rowS)), ent = PROTECT(as_real(entriesS));
  const int m = check_pred_sites("ctx_predict_taper", &v, lp, xp);
  need(LENGTH(row) == m + 1 && XLENGTH(ent) == XLENGTH(col), "ctx_predict_taper", "inconsistent pattern");
  need(XLENGTH(resid) == v.n, "ctx_predict_taper", "the residual must have n elements");
  SEXP out = PROTECT(Rf_allocVector(VECSXP, 2));
  SEXP sto = PROTECT(Rf_allocVector(REALSXP, m)), expl = PROTECT(Rf_allocVector(REALSXP, m));
  int rc = cocons_predict_taper(v.c, m, REAL(lp), REAL(xp), INTEGER(col), INTEGER(row), REAL(ent), XLENGTH(col),
                                REAL(resid), REAL(sto), REAL(expl));
  SET_VECTOR_ELT(out, 0, sto);
  SET_VECTOR_ELT(out, 1, expl);
  UNPROTECT(9);
  raise(rc);
  return out;
}

/* n x k draws L eps for cocoSim (R/sim.R:162-172); eps comes from R's own rnorm */
SEXP _cocons_ctx_sim(SEXP ptr, SEXP epsS) {
  const ctx_view v = view_of(ptr);
  SEXP eps = PROTECT(as_real(epsS));
  need(Rf_isMatrix(eps) && Rf_nrows(eps) == v.n, "ctx_sim", "eps must be an n x k matrix");
  const int n = Rf_nrows(eps), k = Rf_ncols(eps);
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, n, k));
  int rc = cocons_sim(v.c, k, REAL(eps), REAL(out));
  UNPROTECT(2);
  raise(rc);
  return out;
}

/* n x k draws L eps with the kept tapered factor, dense or tiled context (sparse cocoSim, R/sim.R:193-218) */
SEXP _cocons_ctx_sim_taper(SEXP ptr, SEXP epsS) {
  const ctx_view v = view_of(ptr);
  SEXP eps = PROTECT(as_real(epsS));
  need(Rf_isMatrix(eps) && Rf_nrows(eps) == v.n, "ctx_sim_taper", "eps must be an n x k matrix");
  const int n = Rf_nrows(eps), k = Rf_ncols(eps);
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, n, k));
  int rc = cocons_sim_taper(v.c, k, REAL(eps), REAL(out));
  UNPROTECT(2);
  raise(rc);
  return out;
}

/* m x k conditional draws (R/sim.R:87-121) */
SEXP _cocons_ctx_sim_cond(SEXP ptr, SEXP locsPredS, SEXP xPredS, SEXP epsS) {
  const ctx_view v = view_of(ptr);
  SEXP lp = PROTECT(as_real(locsPredS)), xp = PROTECT(as_real(xPredS)), eps = PROTECT(as_real(epsS));
  const int m = check_pred_sites("ctx_sim_cond", &v, lp, xp);
  need(Rf_isMatrix(eps) && Rf_nrows(eps) == m, "ctx_sim_cond", "eps must be an nrow(locs_pred) x k matrix");
  const int k = Rf_ncols(eps);
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, m, k));
  int rc = cocons_sim_cond(v.c, m, REAL(lp), REAL(xp), k, REAL(eps), REAL(out));
  UNPROTECT(4);
  raise(rc);
  return out;
}

/* ---- registration (replaces src/RcppExports.cpp:105-118) -------------------------------- */

static const R_CallMethodDef CallEntries[] = {
    {"_cocons_sumsmoothlone", (DL_FUNC)&_cocons_sumsmoothlone, 3},
    {"_cocons_cov_rns", (DL_FUNC)&_cocons_cov_rns, 4},
    {"_cocons_cov_rns_pred", (DL_FUNC)&_cocons_cov_rns_pred, 6},
    {"_cocons_cov_rns_classic", (DL_FUNC)&_cocons_cov_rns_classic, 3},
    {"_cocons_cov_rns_taper_pred", (DL_FUNC)&_cocons_cov_rns_taper_pred, 8},
    {"_cocons_cov_rns_taper", (DL_FUNC)&_cocons_cov_rns_taper, 6},
    {"_cocons_n2ll_dense", (DL_FUNC)&_cocons_n2ll_dense, 8},
    {"_cocons_ctx_new", (DL_FUNC)&_cocons_ctx_new, 4},
    {"_cocons_ctx_free", (DL_FUNC)&_cocons_ctx_free, 1},
    {"_cocons_ctx_set_z", (DL_FUNC)&_cocons_ctx_set_z, 2},
    {"_cocons_ctx_set_xbetas", (DL_FUNC)&_cocons_ctx_set_xbetas, 2},
    {"_cocons_ctx_n2ll", (DL_FUNC)&_cocons_ctx_n2ll, 7},
    {"_cocons_ctx_new_batch", (DL_FUNC)&_cocons_ctx_new_batch, 5},
    {"_cocons_ctx_n2ll_batch", (DL_FUNC)&_cocons_ctx_n2ll_batch, 7},
    {"_cocons_ctx_factor", (DL_FUNC)&_cocons_ctx_factor, 5},
    {"_cocons_ctx_profile_betas", (DL_FUNC)&_cocons_ctx_profile_betas, 3},
    {"_cocons_ctx_predict", (DL_FUNC)&_cocons_ctx_predict, 4},
    {"_cocons_ctx_set_taper", (DL_FUNC)&_cocons_ctx_set_taper, 4},
    {"_cocons_ctx_new_taper_tiled", (DL_FUNC)&_cocons_ctx_new_taper_tiled, 7},
    {"_cocons_ctx_n2ll_taper", (DL_FUNC)&_cocons_ctx_n2ll_taper, 6},
    {"_cocons_ctx_factor_taper", (DL_FUNC)&_cocons_ctx_factor_taper, 4},
    {"_cocons_ctx_predict_taper", (DL_FUNC)&_cocons_ctx_predict_taper, 7},
    {"_cocons_ctx_sim", (DL_FUNC)&_cocons_ctx_sim, 2},
    {"_cocons_ctx_sim_taper", (DL_FUNC)&_cocons_ctx_sim_taper, 2},
    {"_cocons_ctx_sim_cond", (DL_FUNC)&_cocons_ctx_sim_cond, 4},
    {NULL, NULL, 0}};

void R_init_cocons(DllInfo* dll) {
  R_registerRoutines(dll, NULL, CallEntries, NULL, NULL);
  R_useDynamicSymbols(dll, FALSE);
}
