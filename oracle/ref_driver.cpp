// TEST INFRASTRUCTURE ONLY (oracle/): C entry points around the REFERENCE's own
// dense-covariance source, compiled from where it lies.
//
// `#include "cocons_full.cpp"` below resolves (via -I$(REFERENCE)/src in
// oracle/Makefile; REFERENCE is the reference's source tree, $COCONS_REFERENCE
// or else BASELINE.json's reference_path) to the reference's
// src/cocons_full.cpp, which in turn pulls src/cocons_types.h.  <Rcpp.h> and <boost/math/special_functions/bessel.hpp>
// resolve to the stand-ins under oracle/shim/.  Nothing of the reference is
// copied into this repository; the output (oracle/_ref/libcocons_ref.so) is
// git-ignored and is only ever loaded by tests/, __graft_entry__.smoke() and
// bench.py's CPU-baseline legs.
//
// Wrapped functions (reference file:line):
//   cov_rns          src/cocons_full.cpp:40-321
//   cov_rns_pred     src/cocons_full.cpp:334-471
//   cov_rns_classic  src/cocons_full.cpp:480-594
//   sumsmoothlone    src/cocons_full.cpp:12-30
#include "cocons_full.cpp"

#include <cstring>

namespace {

const char* const kAspectNames[6] = {"std.dev", "scale", "aniso", "tilt", "smooth", "nugget"};

// theta6: six length-p vectors laid out back to back in kAspectNames order
Rcpp::List make_theta(long p, const double* theta6) {
  Rcpp::List th;
  for (int a = 0; a < 6; ++a) th.set(kAspectNames[a], Rcpp::NumericVector(theta6 + a * p, p));
  return th;
}

}  // namespace

extern "C" {

int ref_cov_rns(long n, long p, const double* locs, const double* X, const double* theta6,
                const double* limits, double* out) {
  try {
    Rcpp::List th = make_theta(p, theta6);
    Rcpp::NumericMatrix L(n, 2, locs), Xm(n, p, X);
    Rcpp::NumericVector lim(limits, 2);
    Rcpp::NumericMatrix S = cov_rns(th, L, Xm, lim);
    std::memcpy(out, S.data(), sizeof(double) * (size_t)n * (size_t)n);
    return 0;
  } catch (...) {
    return -1;
  }
}

int ref_cov_rns_pred(long n, long m, long p, const double* locs, const double* locs_pred, const double* X,
                     const double* X_pred, const double* theta6, const double* limits, double* out) {
  try {
    Rcpp::List th = make_theta(p, theta6);
    Rcpp::NumericMatrix L(n, 2, locs), Lp(m, 2, locs_pred), Xm(n, p, X), Xp(m, p, X_pred);
    Rcpp::NumericVector lim(limits, 2);
    Rcpp::NumericMatrix S = cov_rns_pred(th, L, Lp, Xm, Xp, lim);
    std::memcpy(out, S.data(), sizeof(double) * (size_t)n * (size_t)m);
    return 0;
  } catch (...) {
    return -1;
  }
}

int ref_cov_rns_classic(long n, long p, const double* locs, const double* X, const double* theta6, double* out) {
  try {
    Rcpp::List th = make_theta(p, theta6);
    Rcpp::NumericMatrix L(n, 2, locs), Xm(n, p, X);
    Rcpp::NumericMatrix S = cov_rns_classic(th, L, Xm);
    std::memcpy(out, S.data(), sizeof(double) * (size_t)n * (size_t)n);
    return 0;
  } catch (...) {
    return -1;
  }
}

double ref_sumsmoothlone(const double* x, long len, double lambda, double alpha) {
  Rcpp::NumericVector v(x, len);
  return sumsmoothlone(v, lambda, alpha);
}

}  // extern "C"
