// TEST INFRASTRUCTURE ONLY (oracle/): C entry points around the REFERENCE's own
// sparse (tapered) covariance source, compiled from where it lies.
//
// `#include "cocons_taper.cpp"` resolves (via -I$(REFERENCE)/src in
// oracle/Makefile, as in ref_driver.cpp) to the reference's
// src/cocons_taper.cpp.  <Rcpp.h> and the Boost Bessel header resolve to the
// stand-ins under oracle/shim/.  Nothing of
// the reference is copied into this repository; the object is linked into
// oracle/_ref/libcocons_ref.so (git-ignored), which only tests/,
// __graft_entry__.smoke() and bench.py's CPU-baseline legs ever load.
//
// Wrapped functions (reference file:line):
//   cov_rns_taper_pred  src/cocons_taper.cpp:17-139
//   cov_rns_taper       src/cocons_taper.cpp:151-433
// colindices / rowpointers are spam's 1-based CSR arrays, handed over as doubles
// exactly as Rcpp hands them to the reference (it coerces the INTSXP slots).
#include "cocons_taper.cpp"

#include <cstring>

namespace {

const char* const kTaperAspectNames[6] = {"std.dev", "scale", "aniso", "tilt", "smooth", "nugget"};

Rcpp::List make_theta_taper(long p, const double* theta6) {
  Rcpp::List th;
  for (int a = 0; a < 6; ++a) th.set(kTaperAspectNames[a], Rcpp::NumericVector(theta6 + a * p, p));
  return th;
}

}  // namespace

extern "C" {

int ref_cov_rns_taper(long n, long p, const double* locs, const double* X, const double* theta6,
                      const double* limits, const double* colindices, const double* rowpointers, long nnz,
                      double* out) {
  try {
    Rcpp::List th = make_theta_taper(p, theta6);
    Rcpp::NumericMatrix L(n, 2, locs), Xm(n, p, X);
    Rcpp::NumericVector lim(limits, 2), ci(colindices, nnz), rp(rowpointers, n + 1);
    Rcpp::NumericVector v = cov_rns_taper(th, L, Xm, ci, rp, lim);
    for (long k = 0; k < nnz; ++k) out[k] = v[k];
    return 0;
  } catch (...) {
    return -1;
  }
}

int ref_cov_rns_taper_pred(long n, long m, long p, const double* locs, const double* locs_pred, const double* X,
                           const double* X_pred, const double* theta6, const double* limits,
                           const double* colindices, const double* rowpointers, long nnz, double* out) {
  try {
    Rcpp::List th = make_theta_taper(p, theta6);
    Rcpp::NumericMatrix L(n, 2, locs), Lp(m, 2, locs_pred), Xm(n, p, X), Xp(m, p, X_pred);
    Rcpp::NumericVector lim(limits, 2), ci(colindices, nnz), rp(rowpointers, m + 1);
    Rcpp::NumericVector v = cov_rns_taper_pred(th, L, Lp, Xm, Xp, ci, rp, lim);
    for (long k = 0; k < nnz; ++k) out[k] = v[k];
    return 0;
  } catch (...) {
    return -1;
  }
}

}  // extern "C"
