// Sparse (tapered) model: the covariance on the entries of a compactly supported taper pattern,
//   cov_rns_taper       src/cocons_taper.cpp:151-433
//   cov_rns_taper_pred  src/cocons_taper.cpp:17-139
// The pattern is spam's CSR layout (1-based colindices / rowpointers).  This covariance is the
// isotropic member of the family (no anisotropy, no tilt, no global range): per-site range, sigma
// and smoothness only.  One thread per stored entry - a gather over the per-site table, HBM/L2
// bound except for the Bessel tail.  Sinks:
//   * the entry vector itself (what the reference returns to R), and
//   * a scatter of taper[e] * cov[e] into the dense, Morton-ordered lower triangle the blocked
//     Cholesky factors (GetNeg2loglikelihoodTaper, R/neg2loglikelihood.R:20-53, where the
//     reference hands the product to spam's sparse Cholesky), and
//   * a scatter of taper[e] * cov[e] of a block of prediction rows into the dense m x n block the
//     prediction solve works on (cocoPredict sparse branch, R/predict.R:233-251).
// The operation order of the reference is kept through round-to-nearest intrinsics; only the
// transcendental tail (exp, K_nu) differs.
#include <cmath>

#include "../../include/cocons_b200.h"
#include "bessel.cuh"
#include "common.cuh"

namespace cocons {

__device__ __forceinline__ double taper_link_exp(double eta) { return __ddiv_rn(1.0, exp(-eta)); }

// K1t: per-site stage, src/cocons_taper.cpp:54-70 and :195-209.
//   pred_rows = 0: TF_DV = E(std.dev) + E(nugget)          (:229, :243 ...)
//   pred_rows = 1: TF_DV = sigma^2 + E(nugget)             (:91, :111)
__global__ void __launch_bounds__(128) taper_site_stage_kernel(int64_t n, int p, const double* __restrict__ X,
                                                               int64_t ldx, const double* __restrict__ locs,
                                                               int64_t ldl, const double* __restrict__ theta6,
                                                               double lim0, double lim1, int fill_smooth,
                                                               int pred_rows, TaperTable T) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const double* sd = theta6;
  const double* scale = theta6 + p;
  const double* smooth = theta6 + 4 * p;
  const double* nugget = theta6 + 5 * p;
  double e_r = 0, e_sig = 0, e_var = 0, e_nug = 0, e_sm = 0;
  for (int k = 0; k < p; ++k) {
    const double x = X[(int64_t)k * ldx + s];
    e_r = __fma_rn(x, __dmul_rn(2.0, scale[k]), e_r);   // 2 * scale, intercept included
    e_sig = __fma_rn(x, __dmul_rn(0.5, sd[k]), e_sig);  // 0.5 * std.dev
    e_var = __fma_rn(x, sd[k], e_var);
    e_nug = __fma_rn(x, nugget[k], e_nug);
    e_sm = __fma_rn(x, smooth[k], e_sm);
  }
  const double sig = taper_link_exp(e_sig);
  double snu = 0.0;  // stays 0 when the smoothness is fixed (the reference never fills it, :187-199)
  if (fill_smooth)
    snu = __dsqrt_rn(__dadd_rn(__ddiv_rn(__dsub_rn(lim1, lim0), __dadd_rn(1.0, exp(-e_sm))), lim0));
  T.fw(TF_X)[s] = locs[s];
  T.fw(TF_Y)[s] = locs[ldl + s];
  T.fw(TF_R)[s] = taper_link_exp(e_r);
  T.fw(TF_SIG)[s] = sig;
  T.fw(TF_NU)[s] = snu;
  T.fw(TF_DV)[s] = pred_rows ? __dadd_rn(__dmul_rn(sig, sig), taper_link_exp(e_nug))
                             : __dadd_rn(taper_link_exp(e_var), taper_link_exp(e_nug));
}

// one off-diagonal entry (:96-128, :245-264, :384-417); `a` is the row site
template <int MODE>
__device__ __forceinline__ double taper_pair(double ra, double siga, double nua, double rb, double sigb, double nub,
                                             double dx, double dy, double nu_fixed, bool& coincident) {
  const double nu = (MODE == SM_GENERAL || MODE == SM_DEGENERATE) ? __dmul_rn(nua, nub) : nu_fixed;
  const double prefactor =
      __ddiv_rn(__dmul_rn(__dmul_rn(2.0, __dsqrt_rn(ra)), __dsqrt_rn(rb)), __dadd_rn(ra, rb));
  const double avg = __ddiv_rn(__dadd_rn(ra, rb), 2.0);
  const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
  const double Q = __ddiv_rn(__dmul_rn(__dsqrt_rn(__dmul_rn(8.0, nu)), __dsqrt_rn(d2)), __dsqrt_rn(avg));
  coincident = (Q <= 2.220446049250313e-16);
  if (coincident) return 0.0;
  double corr;
  if (MODE == SM_HALF)
    corr = exp(-Q);
  else if (MODE == SM_THREEHALF)
    corr = __dmul_rn(__dadd_rn(1.0, Q), exp(-Q));
  else if (MODE == SM_FIVEHALF)
    corr = __dmul_rn(__dadd_rn(__dadd_rn(1.0, Q), __ddiv_rn(__dmul_rn(Q, Q), 3.0)), exp(-Q));
  else
    corr = (Q < 706.0) ? matern_corr(nu, Q) : matern_corr_tail(nu, Q);
  return __dmul_rn(__dmul_rn(__dmul_rn(prefactor, corr), siga), sigb);
}

// row of CSR entry e: the last r with rowpointers[r] - 1 <= e
__device__ __forceinline__ int64_t taper_row_of(const int* __restrict__ rowpointers, int64_t nrows, int64_t e) {
  int64_t lo = 0, hi = nrows;  // invariant: rowpointers[lo]-1 <= e < rowpointers[hi]-1
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)rowpointers[mid] - 1 <= e)
      lo = mid;
    else
      hi = mid;
  }
  return lo;
}

// K2t.  One thread per stored entry e in [e0, e0 + count).  Rows: table R, columns: table C.
// `square`: rows and columns are the same sites and i == j is the diagonal; otherwise (prediction rows)
// coincidence is exact coordinate equality (:89).  Sinks (TaperSink::kind):
//   TS_VECTOR   out[e] = value                                  (what the reference returns to R)
//   TS_LOWER    A[max(si,sj) + min(si,sj) ld] = taper[e] value  for the entries with i >= j, where
//               si = inv[i] is the site's position in the context's (Morton) ordering
//   TS_ROWS     A[(i - row0) + inv[j] ld] = taper[e] value      (a block of prediction rows x all sites)
//   TS_TILED    as TS_LOWER, into the tile pool of a tiled context: tile (hi / 128, lo / 128) is found by a binary
//               search over the stored tile rows of column lo / 128 (TaperSink::tiles).  Only the instantiations
//               MODE = smoothness mode + kTaperTiled take this sink; the others compile exactly as before.
//   TS_ROWDOT   ONE THREAD PER PATTERN ROW i (count = nrows, e0 = 0): out[i] = sum_e taper[e] value_e A[inv[j_e]] over
//               the row's entries in pattern order (rows from table R at i, columns at inv[j] of the context's table
//               C): the kriging mean C w of the tiled context, w = Sigma^-1 resid.  Instantiation
//               SM_GENERAL + kTaperRowDot of its own.
template <int MODE>
__global__ void __launch_bounds__(256) taper_entries_kernel(int64_t e0, int64_t count, int64_t nrows,
                                                            const int* __restrict__ colindices,
                                                            const int* __restrict__ rowpointers, TaperTable R,
                                                            TaperTable C, int square, double nu_fixed, TaperSink S) {
  constexpr bool kRowDot = MODE >= kTaperRowDot;
  constexpr bool kTiled = MODE >= kTaperTiled && !kRowDot;
  constexpr int kMode = kRowDot ? MODE - kTaperRowDot : (kTiled ? MODE - kTaperTiled : MODE);
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  if constexpr (kRowDot) {
    double s = 0.0;
    for (int64_t e = rowpointers[t] - 1; e < rowpointers[t + 1] - 1; ++e) {
      const int64_t sj = S.inv[colindices[e] - 1];
      const double xi = R.f(TF_X)[t], yi = R.f(TF_Y)[t], xj = C.f(TF_X)[sj], yj = C.f(TF_Y)[sj];
      bool same = (xi == xj && yi == yj);
      double v = 0.0;
      if (!same)
        v = taper_pair<kMode>(R.f(TF_R)[t], R.f(TF_SIG)[t], R.f(TF_NU)[t], C.f(TF_R)[sj], C.f(TF_SIG)[sj],
                              C.f(TF_NU)[sj], __dsub_rn(xi, xj), __dsub_rn(yi, yj), nu_fixed, same);
      if (same) v = R.f(TF_DV)[t];
      s = fma(__dmul_rn(S.taper[e], v), S.A[sj], s);
    }
    S.out[t] = s;
    return;
  }
  const int64_t e = e0 + t;
  const int64_t i = taper_row_of(rowpointers, nrows, e);
  const int64_t j = (int64_t)colindices[e] - 1;
  if ((kTiled || S.kind == TS_LOWER) && i < j) return;  // the dense sink keeps the caller's lower triangle
  // table positions: the context's ordering for resident sites, block-local for prediction rows
  const int64_t si = (kTiled || S.kind == TS_LOWER) ? S.inv[i] : (S.kind == TS_ROWS ? i - S.row0 : i);
  const int64_t sj = (!kTiled && S.kind == TS_VECTOR) ? j : S.inv[j];
  const double xi = R.f(TF_X)[si], yi = R.f(TF_Y)[si];
  const double xj = C.f(TF_X)[sj], yj = C.f(TF_Y)[sj];
  double v = 0.0;
  bool same = square ? (i == j) : (xi == xj && yi == yj);
  if (!same)
    v = taper_pair<kMode>(R.f(TF_R)[si], R.f(TF_SIG)[si], R.f(TF_NU)[si], C.f(TF_R)[sj], C.f(TF_SIG)[sj],
                         C.f(TF_NU)[sj], __dsub_rn(xi, xj), __dsub_rn(yi, yj), nu_fixed, same);
  if (same) v = R.f(TF_DV)[si];
  if (kTiled) {
    const int64_t hi = si > sj ? si : sj, lo = si > sj ? sj : si;
    const int64_t I = hi / kTile, J = lo / kTile, T = S.ld, nst = S.row0;
    const int64_t* rows = S.tiles + T + 1;
    int64_t a = S.tiles[J], b = S.tiles[J + 1] - 1;  // every tile of the pattern is stored: rows[a..b] holds I
    while (a < b) {
      const int64_t mid = (a + b) >> 1;
      if (rows[mid] < I)
        a = mid + 1;
      else
        b = mid;
    }
    const int64_t ld = S.tiles[T + 1 + 2 * nst + J];
    S.A[rows[nst + a] + (lo % kTile) * ld + hi % kTile] = __dmul_rn(S.taper[e], v);
  } else if (S.kind == TS_VECTOR) {
    S.out[e] = v;
  } else if (S.kind == TS_LOWER) {
    const int64_t hi = si > sj ? si : sj, lo = si > sj ? sj : si;
    S.A[hi + lo * S.ld] = __dmul_rn(S.taper[e], v);
  } else {
    S.A[si + sj * S.ld] = __dmul_rn(S.taper[e], v);
  }
}

// unit diagonal in the padding rows of the dense sink
__global__ void taper_pad_diag_kernel(int64_t n, int64_t n_pad, double* __restrict__ A, int64_t ld) {
  const int64_t s = n + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n_pad) A[s + s * ld] = 1.0;
}

void launch_taper_site_stage(int64_t n, int p, const double* dX, int64_t ldx, const double* dlocs, int64_t ldl,
                             const double* dtheta6, double lim0, double lim1, int mode, int pred_rows, TaperTable T,
                             cudaStream_t st) {
  note_launch();
  taper_site_stage_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(n, p, dX, ldx, dlocs, ldl, dtheta6, lim0, lim1,
                                                                       mode == SM_GENERAL, pred_rows, T);
}

void launch_taper_entries(int64_t e0, int64_t count, int64_t nrows, const int* dcol, const int* drow, TaperTable R,
                          TaperTable C, int square, int mode, double nu_fixed, TaperSink S, cudaStream_t st) {
  if (count <= 0) return;
  const unsigned blocks = (unsigned)((count + 255) / 256);
  note_launch();
#define COCONS_TAPER_LAUNCH(M) \
  taper_entries_kernel<M><<<blocks, 256, 0, st>>>(e0, count, nrows, dcol, drow, R, C, square, nu_fixed, S)
  switch (mode + (S.kind == TS_TILED ? kTaperTiled : (S.kind == TS_ROWDOT ? kTaperRowDot : 0))) {
    case SM_HALF: COCONS_TAPER_LAUNCH(SM_HALF); break;
    case SM_THREEHALF: COCONS_TAPER_LAUNCH(SM_THREEHALF); break;
    case SM_FIVEHALF: COCONS_TAPER_LAUNCH(SM_FIVEHALF); break;
    case SM_DEGENERATE: COCONS_TAPER_LAUNCH(SM_DEGENERATE); break;
    case SM_HALF + kTaperTiled: COCONS_TAPER_LAUNCH(SM_HALF + kTaperTiled); break;
    case SM_THREEHALF + kTaperTiled: COCONS_TAPER_LAUNCH(SM_THREEHALF + kTaperTiled); break;
    case SM_FIVEHALF + kTaperTiled: COCONS_TAPER_LAUNCH(SM_FIVEHALF + kTaperTiled); break;
    case SM_DEGENERATE + kTaperTiled: COCONS_TAPER_LAUNCH(SM_DEGENERATE + kTaperTiled); break;
    case SM_GENERAL + kTaperTiled: COCONS_TAPER_LAUNCH(SM_GENERAL + kTaperTiled); break;
    case SM_GENERAL + kTaperRowDot: COCONS_TAPER_LAUNCH(SM_GENERAL + kTaperRowDot); break;
    default: COCONS_TAPER_LAUNCH(SM_GENERAL); break;
  }
#undef COCONS_TAPER_LAUNCH
}

void launch_taper_pad_diag(int64_t n, int64_t n_pad, double* A, int64_t ld, cudaStream_t st) {
  if (n_pad <= n) return;
  note_launch();
  taper_pad_diag_kernel<<<(unsigned)((n_pad - n + 127) / 128), 128, 0, st>>>(n, n_pad, A, ld);
}

}  // namespace cocons
