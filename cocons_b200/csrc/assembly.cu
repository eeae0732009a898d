// Covariance assembly on the device: the per-site stage (K1) and the tiled
// pairwise kernels (K2) that replace the O(n^2) loops of
//   cov_rns          src/cocons_full.cpp:114-317
//   cov_rns_pred     src/cocons_full.cpp:407-468
//   cov_rns_classic  src/cocons_full.cpp:529-591
// FP64 throughout.  The pair geometry (local-kernel averaging, determinant,
// scaled distance Q) keeps the reference's operation order - including its
// difference-of-products helper (src/cocons_types.h:49-54) - through explicit
// round-to-nearest intrinsics, because the entry is ~exp(-Q) and an error in Q
// is amplified Q-fold.  Only the transcendental tail (exp, K_nu) differs.
#include <algorithm>
#include <cmath>
#include <vector>

#include "../../include/cocons_b200.h"
#include "bessel.cuh"
#include "common.cuh"

namespace cocons {

// ---------------------------------------------------------------------------
// K1: per-site stage.  One thread per site; every linear predictor is the
// sequential fma chain of src/cocons_types.h:12-17 over the site's row of X.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double link_exp(double eta) { return __ddiv_rn(1.0, exp(-eta)); }

// BATCH = 1: blockIdx.y is the point of a batch, with its own theta (7 p apart) and site table (SF_COUNT tables apart)
template <int BATCH>
__global__ void __launch_bounds__(128) site_stage_kernel(int64_t n, int64_t n_fill, int p, const double* __restrict__ X,
                                                         int64_t ldx, const double* __restrict__ locs, int64_t ldl,
                                                         const double* __restrict__ theta6, double lim0, double lim1,
                                                         int mode, SiteTable T) {
  if constexpr (BATCH) {
    theta6 += (int64_t)blockIdx.y * 7 * p;
    T.base += (int64_t)blockIdx.y * SF_COUNT * T.stride;
  }
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_fill) return;
  if (s >= n) {  // padding sites: never used by a real pair
    for (int f = 0; f < SF_COUNT; ++f) T.fw(f)[s] = 0.0;
    T.fw(SF_DV)[s] = 1.0;
    return;
  }
  const double* sd = theta6;
  const double* scale = theta6 + p;
  const double* aniso = theta6 + 2 * p;
  const double* tilt = theta6 + 3 * p;
  const double* smooth = theta6 + 4 * p;
  const double* nugget = theta6 + 5 * p;
  double e_tilt = 0, e_r = 0, e_a = 0, e_d = 0, e_sig = 0, e_nug = 0, e_var = 0, e_sm = 0;
  for (int k = 0; k < p; ++k) {
    const double x = X[(int64_t)k * ldx + s];
    const double sj = (k == 0) ? 0.0 : scale[k];         // scale_je       :64
    const double two_sj = __dmul_rn(2.0, sj);            // 2 * scale_je   :101
    const double root = __dadd_rn(two_sj, aniso[k]);     // sqrt_vector    :66
    const double half_sd = __dmul_rn(0.5, sd[k]);        //                :104
    e_tilt = __fma_rn(x, tilt[k], e_tilt);
    e_r = __fma_rn(x, two_sj, e_r);
    e_a = __fma_rn(x, aniso[k], e_a);
    e_d = __fma_rn(x, root, e_d);
    e_sig = __fma_rn(x, half_sd, e_sig);
    e_nug = __fma_rn(x, nugget[k], e_nug);
    e_var = __fma_rn(x, sd[k], e_var);
    e_sm = __fma_rn(x, smooth[k], e_sm);
  }
  const double t = __ddiv_rn(kPi, __dadd_rn(1.0, exp(-e_tilt)));  // types.h:46
  const double r = link_exp(e_r);
  const double a = link_exp(e_a);
  const double D = link_exp(e_d);
  const double cs = cos(t), sn = sin(t);
  const double a2 = __dmul_rn(a, a);
  const double ra = __dmul_rn(r, a);
  const double p22 = __dmul_rn(r, a2);
  const double p12 = __dmul_rn(ra, cs);
  double snu = 0.0;
  if (mode == SM_CLASSIC)
    snu = link_exp(e_sm);  // :524
  else if (mode == SM_GENERAL)
    snu = __dsqrt_rn(__dadd_rn(__ddiv_rn(__dsub_rn(lim1, lim0), __dadd_rn(1.0, exp(-e_sm))), lim0));  // :93
  T.fw(SF_X)[s] = locs[s];
  T.fw(SF_Y)[s] = locs[ldl + s];
  T.fw(SF_R)[s] = r;
  T.fw(SF_A2)[s] = a2;
  T.fw(SF_RA)[s] = ra;
  T.fw(SF_CS)[s] = cs;
  T.fw(SF_P22)[s] = p22;
  T.fw(SF_E22)[s] = __fma_rn(r, a2, -p22);
  T.fw(SF_P12)[s] = p12;
  T.fw(SF_E12)[s] = __fma_rn(ra, cs, -p12);
  T.fw(SF_NU)[s] = snu;
  // amplitude factor of the site: sigma_i sqrt(D_i sin t_i).  The reference forms
  // corr sigma_i sigma_j sqrt(D_i sin t_i D_j sin t_j) / sqrt(det) per pair (:295-297); hoisting the square root
  // to the site moves an entry by a few ulp (no amplification here, unlike Q) and takes two square roots and a
  // division out of the pair loop.  SF_SIG / SF_W stay in the table for the entries that end up near the
  // subnormal range, where the reference's own sequence of roundings is followed (pair_cov).
  const double sig = link_exp(e_sig), w = __dmul_rn(D, sn);
  T.fw(SF_SIG)[s] = sig;
  T.fw(SF_W)[s] = w;
  T.fw(SF_AMP)[s] = __dmul_rn(sig, __dsqrt_rn(w));
  T.fw(SF_DV)[s] = __dadd_rn(link_exp(e_var), link_exp(e_nug));  // :111
}

// ---------------------------------------------------------------------------
// Pair arithmetic.  `a` plays the reference's "ii" role (first operand of its
// kahan() calls), `b` the "jj" role, whose products arrive pre-split as
// (P, e) = (rnd(c d), c d - rnd(c d)).
// ---------------------------------------------------------------------------
struct SiteA {
  double x, y, r, a2, ra, cs, nu, amp, dv;
};
struct SiteB {
  double x, y, r, p22, e22, p12, e12, nu, amp;
};

// Correlations below this go through `slow_amp` (the reference's operation order on sigma and D sin t read back
// from the site table): their entries may be subnormal, where every intermediate rounding of the reference shows.
constexpr double kTinyCorr = 1e-250;

template <int MODE, class SlowAmp>
__device__ __forceinline__ double pair_cov(const SiteA& a, const SiteB& b, double global_range, double nu_fixed,
                                           bool& coincident, SlowAmp slow_amp, const double* exp_tab = nullptr) {
  // sigma11, sigma22, sigma12 of the averaged kernel matrix (:260-268)
  const double s11 = __dmul_rn(__dadd_rn(a.r, b.r), 0.5);
  const double s22 = __dmul_rn(__dadd_rn(__fma_rn(a.r, a.a2, b.p22), b.e22), 0.5);
  const double s12 = __dmul_rn(__dadd_rn(__fma_rn(a.ra, a.cs, b.p12), b.e12), 0.5);
  // det = kahan(s11, s22, s12, s12) (:270)
  const double cd = __dmul_rn(s12, s12);
  const double det = __dsub_rn(__fma_rn(s11, s22, -cd), __fma_rn(s12, s12, -cd));
  const double dx = __dsub_rn(a.x, b.x), dy = __dsub_rn(a.y, b.y);
  double nu;
  if (MODE == SM_GENERAL || MODE == SM_DEGENERATE)
    nu = __dmul_rn(a.nu, b.nu);  // :274
  else if (MODE == SM_CLASSIC)
    nu = __ddiv_rn(__dadd_rn(a.nu, b.nu), 2.0);  // :554
  else
    nu = nu_fixed;
  // quadratic form: fma(kahan(s22, dx^2, -s11, dy^2), 1, -2 s12 dx dy) (:277-281)
  const double dx2 = __dmul_rn(dx, dx), dy2 = __dmul_rn(dy, dy);
  const double ns11 = -s11;
  const double cd2 = __dmul_rn(ns11, dy2);
  const double k1 = __dsub_rn(__fma_rn(s22, dx2, -cd2), __fma_rn(ns11, dy2, -cd2));
  const double cross = __dmul_rn(__dmul_rn(__dmul_rn(-2.0, s12), dx), dy);
  const double quad = __dadd_rn(k1, cross);
  const double Q = __dmul_rn(__dsqrt_rn(__ddiv_rn(__dmul_rn(8.0, nu), __dmul_rn(global_range, det))),
                             __dsqrt_rn(quad));
  coincident = (Q <= 2.220446049250313e-16);  // :284
  if (coincident) return 0.0;
  double corr;
  if (MODE == SM_HALF) {
    corr = exp(-Q);  // :150
  } else if (MODE == SM_THREEHALF) {
    corr = __dmul_rn(__dadd_rn(1.0, Q), exp(-Q));  // :196
  } else if (MODE == SM_FIVEHALF) {
    corr = __dmul_rn(__dadd_rn(__dadd_rn(1.0, Q), __ddiv_rn(__dmul_rn(Q, Q), 3.0)), exp(-Q));  // :242
  } else {
    corr = (Q < 706.0) ? matern_corr(nu, Q, exp_tab) : matern_corr_tail(nu, Q);  // :291-305
  }
  // corr * sigma_i * sigma_j * sqrt(D_i sin t_i D_j sin t_j) / sqrt(det) (:295-297) with the per-site parts hoisted
  if (!(fabs(corr) >= kTinyCorr)) return slow_amp(corr, det);
  return __dmul_rn(__dmul_rn(corr, __dmul_rn(a.amp, b.amp)), rsqrt(det));
}

// the amplitude in the reference's order, left to right (:295-297); sa / wa belong to the "ii" site
__device__ __noinline__ double amp_reference_order(double corr, double det, double sa, double sb, double wa,
                                                   double wb) {
  const double amp = __dmul_rn(__dmul_rn(corr, sa), sb);
  return __ddiv_rn(__dmul_rn(amp, __dsqrt_rn(__dmul_rn(wa, wb))), __dsqrt_rn(det));
}

// ---------------------------------------------------------------------------
// K2a: lower-triangle assembly, 128 x 128 tiles, one thread per row of the
// tile, the 128 column sites staged in shared memory and broadcast.  A warp
// covers 32 consecutive rows of one column at a time, so its 32 stores form
// one 256-byte segment of the column-major matrix.  Column sites are the lower
// index => the reference's "ii" role.
// ---------------------------------------------------------------------------
constexpr int kAsmTile = 128;

__device__ __forceinline__ void tri_decode(int64_t t, int& tr, int& tc) {
  int r = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while ((int64_t)(r + 1) * (r + 2) / 2 <= t) ++r;
  while ((int64_t)r * (r + 1) / 2 > t) --r;
  tr = r;
  tc = (int)(t - (int64_t)r * (r + 1) / 2);
}

#ifndef COCONS_ASM_MINBLOCKS
#define COCONS_ASM_MINBLOCKS 8
#endif
// KMODE = mode + kAsmBatch: the lower triangle of matrix blockIdx.y of a batch (launch_assemble_lower_batch); `ld`
// carries the device address of the batch's global ranges, the matrices are T.stride x T.stride
template <int KMODE>
__global__ void __launch_bounds__(kAsmTile, COCONS_ASM_MINBLOCKS) assemble_lower_kernel(int64_t n, int64_t n_out, SiteTable T,
                                                                  double global_range, double nu_fixed,
                                                                  double* __restrict__ C, int64_t ld, int col_tile0,
                                                                  int slab) {
  constexpr int MODE = KMODE % kAsmBatch;
  if constexpr (KMODE >= kAsmBatch) {
    global_range = reinterpret_cast<const double*>(ld)[blockIdx.y];
    ld = T.stride;
    T.base += (int64_t)blockIdx.y * SF_COUNT * T.stride;
    C += (int64_t)blockIdx.y * ld * ld;
  }
  // slab == 0: C is the whole matrix, blockIdx.x runs over its lower-triangle tiles.
  // slab == 1: C holds only the tile columns [col_tile0, col_tile0 + gridDim.y) (a column panel of a
  //            distributed matrix); blockIdx.x runs over the tile rows from col_tile0 down.
  __shared__ double cs[9][kAsmTile];
  __shared__ double etab[kAsmTile];  // 2^(j/128) of the node exponential (bessel.cuh)
  __shared__ int corig[kAsmTile];
  static_assert(kAsmTile == 128, "one table entry per thread");
  int tr, tc;
  if (slab >= 2) {
    // slab = 2 + 16 (world + 64 rank): C holds ALL column panels of one rank of the block-cyclic layout (csrc/dist.cu:
    // 4-tile panels dealt in a snake), back to back; blockIdx.y is the local tile column, blockIdx.x the tile row.
    // One launch per evaluation instead of one per panel (98 launches of ~1.3 waves each at n = 50 000).
    const int world = (slab >> 4) & 63, rank = slab >> 10;
    const int lc = blockIdx.y, lp = lc >> 2;
    const int K = lp * world + ((lp & 1) ? world - 1 - rank : rank);
    tc = K * 4 + (lc & 3);
    tr = blockIdx.x;
    if (tr < tc || (int64_t)tc * kAsmTile >= n_out) return;
    C += ((int64_t)lc - tc) * kAsmTile * ld;
  } else if (slab) {
    tr = col_tile0 + blockIdx.x;
    tc = col_tile0 + blockIdx.y;
    if (tr < tc) return;
    C -= (int64_t)col_tile0 * kAsmTile * ld;
  } else {
    tri_decode(blockIdx.x, tr, tc);
  }
  const int tid = threadIdx.x;
  const int64_t I = (int64_t)tr * kAsmTile + tid;
  const int64_t J0 = (int64_t)tc * kAsmTile;
  {
    const int64_t J = J0 + tid;
    const bool ok = J < n;
    cs[0][tid] = ok ? T.f(SF_X)[J] : 0.0;
    cs[1][tid] = ok ? T.f(SF_Y)[J] : 0.0;
    cs[2][tid] = ok ? T.f(SF_R)[J] : 1.0;
    cs[3][tid] = ok ? T.f(SF_A2)[J] : 1.0;
    cs[4][tid] = ok ? T.f(SF_RA)[J] : 1.0;
    cs[5][tid] = ok ? T.f(SF_CS)[J] : 0.0;
    cs[6][tid] = ok ? T.f(SF_NU)[J] : 1.0;
    cs[7][tid] = ok ? T.f(SF_AMP)[J] : 0.0;
    cs[8][tid] = ok ? T.f(SF_DV)[J] : 1.0;
    corig[tid] = (ok && T.orig) ? T.orig[J] : (int)J;
    etab[tid] = kExp2Tab[tid];
  }
  SiteB b;
  double dvI = 1.0;
  int origI = (int)I;
  const bool rowok = I < n;
  if (rowok) {
    b.x = T.f(SF_X)[I];
    b.y = T.f(SF_Y)[I];
    b.r = T.f(SF_R)[I];
    b.p22 = T.f(SF_P22)[I];
    b.e22 = T.f(SF_E22)[I];
    b.p12 = T.f(SF_P12)[I];
    b.e12 = T.f(SF_E12)[I];
    b.nu = T.f(SF_NU)[I];
    b.amp = T.f(SF_AMP)[I];
    dvI = T.f(SF_DV)[I];
    if (T.orig) origI = T.orig[I];
  } else {
    b.x = b.y = 0.0;
    b.r = b.p22 = b.p12 = 1.0;
    b.e22 = b.e12 = 0.0;
    b.nu = 1.0;
    b.amp = 0.0;
  }
  __syncthreads();
  if (I >= n_out) return;
  const bool diag_tile = (tr == tc);
  // small problems: gridDim.z CTAs share a tile, each taking a slice of its 128 columns, so that a
  // handful of tiles still spreads over all SMs
  const int cw = kAsmTile / (int)gridDim.z;
  const int jlo = (int)blockIdx.z * cw;
  const int jend = min(diag_tile ? tid : (kAsmTile - 1), jlo + cw - 1);
  for (int j = jlo; j <= jend; ++j) {
    const int64_t J = J0 + j;
    if (J >= n_out) break;
    double v;
    if (I == J) {
      v = dvI;  // :110-112
    } else if (!rowok || J >= n) {
      v = 0.0;  // padding: identity block
    } else {
      SiteA a;
      a.x = cs[0][j];
      a.y = cs[1][j];
      a.r = cs[2][j];
      a.a2 = cs[3][j];
      a.ra = cs[4][j];
      a.cs = cs[5][j];
      a.nu = cs[6][j];
      a.amp = cs[7][j];
      a.dv = cs[8][j];
      bool coincident;
      v = pair_cov<MODE>(a, b, global_range, nu_fixed, coincident, [&](double corr, double det) {
        return amp_reference_order(corr, det, T.f(SF_SIG)[J], T.f(SF_SIG)[I], T.f(SF_W)[J], T.f(SF_W)[I]);
      }, etab);
      // :284-286 - the value of the lower caller-order index of the pair
      if (coincident) v = (corig[j] < origI) ? a.dv : dvI;
    }
    C[J * ld + I] = v;
    if (diag_tile && j < tid) C[I * ld + J] = v;  // keep diagonal tiles fully symmetric
  }
}

// ---------------------------------------------------------------------------
// K2b: rectangular cross-covariance (prediction sites x training sites),
// always the general Bessel branch; prediction sites are rows and take the
// "ii" role (src/cocons_full.cpp:407-468).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kAsmTile) assemble_cross_kernel(int64_t m, int64_t n, SiteTable P, SiteTable T,
                                                                  double global_range, double* __restrict__ C,
                                                                  int64_t ld) {
  __shared__ double cs[9][kAsmTile];
  const int tid = threadIdx.x;
  const int64_t I = (int64_t)blockIdx.x * kAsmTile + tid;
  const int64_t J0 = (int64_t)blockIdx.y * kAsmTile;
  {
    const int64_t J = J0 + tid;
    const bool ok = J < n;
    cs[0][tid] = ok ? T.f(SF_X)[J] : 0.0;
    cs[1][tid] = ok ? T.f(SF_Y)[J] : 0.0;
    cs[2][tid] = ok ? T.f(SF_R)[J] : 1.0;
    cs[3][tid] = ok ? T.f(SF_P22)[J] : 1.0;
    cs[4][tid] = ok ? T.f(SF_E22)[J] : 0.0;
    cs[5][tid] = ok ? T.f(SF_P12)[J] : 1.0;
    cs[6][tid] = ok ? T.f(SF_E12)[J] : 0.0;
    cs[7][tid] = ok ? T.f(SF_NU)[J] : 1.0;
    cs[8][tid] = ok ? T.f(SF_AMP)[J] : 0.0;
  }
  SiteA a;
  const bool rowok = I < m;
  if (rowok) {
    a.x = P.f(SF_X)[I];
    a.y = P.f(SF_Y)[I];
    a.r = P.f(SF_R)[I];
    a.a2 = P.f(SF_A2)[I];
    a.ra = P.f(SF_RA)[I];
    a.cs = P.f(SF_CS)[I];
    a.nu = P.f(SF_NU)[I];
    a.amp = P.f(SF_AMP)[I];
    a.dv = P.f(SF_DV)[I];
  }
  __syncthreads();
  if (!rowok) return;
  const int jend = (int)min((int64_t)kAsmTile, n - J0);
  for (int j = 0; j < jend; ++j) {
    SiteB b;
    b.x = cs[0][j];
    b.y = cs[1][j];
    b.r = cs[2][j];
    b.p22 = cs[3][j];
    b.e22 = cs[4][j];
    b.p12 = cs[5][j];
    b.e12 = cs[6][j];
    b.nu = cs[7][j];
    b.amp = cs[8][j];
    double v;
    if (a.x == b.x && a.y == b.y) {  // :410
      v = a.dv;
    } else {
      bool coincident;
      v = pair_cov<SM_GENERAL>(a, b, global_range, 0.0, coincident, [&](double corr, double det) {
        return amp_reference_order(corr, det, P.f(SF_SIG)[I], T.f(SF_SIG)[J0 + j], P.f(SF_W)[I], T.f(SF_W)[J0 + j]);
      });
      if (coincident) v = a.dv;  // :440-442
    }
    C[(J0 + j) * ld + I] = v;
  }
}

// mirror the strict lower triangle into the upper one (full symmetric output of cov_rns)
__global__ void __launch_bounds__(256) symmetrize_kernel(int64_t n, double* __restrict__ C, int64_t ld) {
  __shared__ double tile[32][33];
  const int bx = blockIdx.x, by = blockIdx.y;  // tile (row block by, col block bx), by >= bx
  if (by < bx) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int k = ty; k < 32; k += 8) {
    const int64_t i = (int64_t)by * 32 + tx, j = (int64_t)bx * 32 + k;
    tile[k][tx] = (i < n && j < n) ? C[j * ld + i] : 0.0;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    // write element (row = bx*32 + tx, col = by*32 + k) = lower(by*32 + k, bx*32 + tx)
    const int64_t i = (int64_t)bx * 32 + tx, j = (int64_t)by * 32 + k;
    if (i < n && j < n && i < j) C[j * ld + i] = tile[tx][k];
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------

// src/cocons_full.cpp:77-96 + src/cocons_types.h:56-70
int smooth_mode_for(int par, int p, const double* theta6, const double* limits, double* nu_fixed) {
  *nu_fixed = 0.0;
  if (par == COCONS_PAR_CLASSIC) return SM_CLASSIC;
  const double* smooth = theta6 + 4 * (int64_t)p;
  bool slopes_zero = true;
  for (int k = 1; k < p; ++k)
    if (smooth[k] != 0) slopes_zero = false;
  if (slopes_zero && limits[0] == limits[1]) {
    *nu_fixed = limits[0];
    if (std::fabs(limits[0] - 0.5) < 1e-6) return SM_HALF;
    if (std::fabs(limits[0] - 1.5) < 1e-6) return SM_THREEHALF;
    if (std::fabs(limits[0] - 2.5) < 1e-6) return SM_FIVEHALF;
    return SM_DEGENERATE;
  }
  return SM_GENERAL;
}

template <int BATCH>
static void launch_site_stage_k(dim3 grid, int64_t n, int64_t n_fill, int p, const double* dX, int64_t ldx,
                                const double* dlocs, int64_t ldl, const double* dtheta6, double lim0, double lim1,
                                int mode, SiteTable T, cudaStream_t st) {
  site_stage_kernel<BATCH><<<grid, 128, 0, st>>>(n, n_fill, p, dX, ldx, dlocs, ldl, dtheta6, lim0, lim1, mode, T);
}

void launch_site_stage(int64_t n, int64_t n_fill, int p, const double* dX, int64_t ldx, const double* dlocs,
                       int64_t ldl, const double* dtheta6, double lim0, double lim1, int mode, SiteTable T,
                       cudaStream_t st, int batch) {
  const int threads = 128;
  const unsigned blocks = (unsigned)((n_fill + threads - 1) / threads);
  // the degenerate mode leaves smooth_vector at zero, exactly as the reference does
  note_launch();
  if (batch > 0)
    launch_site_stage_k<1>(dim3(blocks, (unsigned)batch), n, n_fill, p, dX, ldx, dlocs, ldl, dtheta6, lim0, lim1, mode,
                           T, st);
  else
    launch_site_stage_k<0>(dim3(blocks), n, n_fill, p, dX, ldx, dlocs, ldl, dtheta6, lim0, lim1, mode, T, st);
}

template <int OFF>
static void launch_assemble_any(int64_t n, int64_t n_out, SiteTable T, double global_range, double nu_fixed, int mode,
                                double* C, int64_t ld, int col_tile0, int slab, dim3 grid, cudaStream_t st);

// ~1200 CTAs fit the GPU at once; measured: holes (990 tiles) 2 / 4 / 8 / 16 / 32 slices -> 1.15 / 0.99 / 0.91 /
// 0.87 / 0.89 ms, stripes (4465 tiles) -> 3.58 / 3.45 / 3.41 / 3.46 / 3.59 ms
static unsigned assemble_slices(int64_t tiles) {
  unsigned slices = tiles < 1500 ? 16u : (tiles < 6000 ? 8u : (tiles < 9600 ? 4u : 1u));
  if (const char* e = getenv("COCONS_ASM_SLICES")) {  // experiment knob: 1, 2, 4, 8, 16, 32
    const int v = atoi(e);
    if (v >= 1 && v <= 32 && (v & (v - 1)) == 0) slices = (unsigned)v;
  }
  return slices;
}

void launch_assemble_lower(int64_t n, int64_t n_out, SiteTable T, double global_range, double nu_fixed, int mode,
                           double* C, int64_t ld, cudaStream_t st) {
  const int64_t nt = (n_out + kAsmTile - 1) / kAsmTile;
  const int64_t tiles = nt * (nt + 1) / 2;
  launch_assemble_any<0>(n, n_out, T, global_range, nu_fixed, mode, C, ld, 0, 0,
                         dim3((unsigned)tiles, 1, assemble_slices(tiles)), st);
}

void launch_assemble_lower_batch(int64_t n, int64_t n_out, SiteTable T, const double* dranges, double nu_fixed,
                                 int mode, double* C, int batch, cudaStream_t st) {
  const int64_t nt = (n_out + kAsmTile - 1) / kAsmTile;
  const int64_t tiles = nt * (nt + 1) / 2;
  launch_assemble_any<kAsmBatch>(n, n_out, T, 0.0, nu_fixed, mode, C, (int64_t)(uintptr_t)dranges, 0, 0,
                                 dim3((unsigned)tiles, (unsigned)batch, assemble_slices(tiles)), st);
}

// column panel [col_tile0, col_tile0 + ncol_tiles) of the lower triangle into a slab whose first
// column is tile column col_tile0 (rows keep their global index, leading dimension ld)
void launch_assemble_panel(int64_t n, int64_t n_out, SiteTable T, double global_range, double nu_fixed, int mode,
                           double* slab, int64_t ld, int col_tile0, int ncol_tiles, cudaStream_t st) {
  const int64_t nt = (n_out + kAsmTile - 1) / kAsmTile;
  launch_assemble_any<0>(n, n_out, T, global_range, nu_fixed, mode, slab, ld, col_tile0, 1,
                      dim3((unsigned)(nt - col_tile0), (unsigned)ncol_tiles), st);
}

// all column panels of one rank of the block-cyclic layout (nlocal panels of 4 tile columns, back to back in `slab`)
void launch_assemble_cyclic(int64_t n, int64_t n_out, SiteTable T, double global_range, double nu_fixed, int mode,
                            double* slab, int64_t ld, int world, int rank, int64_t nlocal, cudaStream_t st) {
  const int64_t nt = (n_out + kAsmTile - 1) / kAsmTile;
  if (nlocal <= 0 || world > 63) return;
  launch_assemble_any<0>(n, n_out, T, global_range, nu_fixed, mode, slab, ld, 0, 2 | (world << 4) | (rank << 10),
                      dim3((unsigned)nt, (unsigned)(nlocal * 4)), st);
}

// OFF = kAsmBatch: the batched instantiations
template <int OFF>
static void launch_assemble_any(int64_t n, int64_t n_out, SiteTable T, double global_range, double nu_fixed, int mode,
                                double* C, int64_t ld, int col_tile0, int slab, dim3 grid, cudaStream_t st) {
  note_launch();
#define COCONS_ASM_CASE(M)                                                                          \
  case M:                                                                                           \
    assemble_lower_kernel<M + OFF><<<grid, kAsmTile, 0, st>>>(n, n_out, T, global_range, nu_fixed, C, ld, col_tile0, \
                                                              slab);                                 \
    break;
  switch (mode) {
    COCONS_ASM_CASE(SM_GENERAL)
    COCONS_ASM_CASE(SM_HALF)
    COCONS_ASM_CASE(SM_THREEHALF)
    COCONS_ASM_CASE(SM_FIVEHALF)
    COCONS_ASM_CASE(SM_CLASSIC)
    COCONS_ASM_CASE(SM_DEGENERATE)
  }
#undef COCONS_ASM_CASE
}

void launch_assemble_cross(int64_t m, int64_t n, SiteTable Tpred, SiteTable Ttrain, double global_range, double* C,
                           int64_t ld, cudaStream_t st) {
  dim3 grid((unsigned)((m + kAsmTile - 1) / kAsmTile), (unsigned)((n + kAsmTile - 1) / kAsmTile));
  note_launch();
  assemble_cross_kernel<<<grid, kAsmTile, 0, st>>>(m, n, Tpred, Ttrain, global_range, C, ld);
}

void launch_symmetrize(int64_t n, double* C, int64_t ld, cudaStream_t st) {
  const unsigned nb = (unsigned)((n + 31) / 32);
  note_launch();
  symmetrize_kernel<<<dim3(nb, nb), 256, 0, st>>>(n, C, ld);
}

// Morton (Z-order) permutation of the sites: perm[s] = caller index of the
// s-th site along the curve.  Spatially close sites become index-close, so a
// warp of the assembly kernel (32 consecutive rows x one column) sees nearly
// equal Q and takes one Bessel branch.
void morton_order(int64_t n, const double* locs, int64_t* perm) {
  double lo[2] = {INFINITY, INFINITY}, hi[2] = {-INFINITY, -INFINITY};
  for (int d = 0; d < 2; ++d)
    for (int64_t i = 0; i < n; ++i) {
      const double v = locs[d * n + i];
      if (v < lo[d]) lo[d] = v;
      if (v > hi[d]) hi[d] = v;
    }
  std::vector<std::pair<uint64_t, int64_t>> key((size_t)n);
  auto spread = [](uint64_t v) {
    v &= 0xFFFFFFFFull;
    v = (v | (v << 16)) & 0x0000FFFF0000FFFFull;
    v = (v | (v << 8)) & 0x00FF00FF00FF00FFull;
    v = (v | (v << 4)) & 0x0F0F0F0F0F0F0F0Full;
    v = (v | (v << 2)) & 0x3333333333333333ull;
    v = (v | (v << 1)) & 0x5555555555555555ull;
    return v;
  };
  for (int64_t i = 0; i < n; ++i) {
    uint64_t q[2];
    for (int d = 0; d < 2; ++d) {
      const double span = hi[d] - lo[d];
      double u = (span > 0 && std::isfinite(span)) ? (locs[d * n + i] - lo[d]) / span : 0.0;
      if (!(u >= 0)) u = 0;
      if (u > 1) u = 1;
      q[d] = (uint64_t)(u * 4294967295.0);
    }
    key[(size_t)i] = {spread(q[0]) | (spread(q[1]) << 1), i};
  }
  std::sort(key.begin(), key.end());
  for (int64_t i = 0; i < n; ++i) perm[i] = key[(size_t)i].second;
}

}  // namespace cocons
