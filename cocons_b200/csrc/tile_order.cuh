// Banded, lower-only rasterisation of the 128-row tiles of a C -= A B^T update, shared by the DMMA GEMM
// (chol.cu) and the split-int8 update (syrk_i8.cu).
#ifndef COCONS_TILE_ORDER_CUH
#define COCONS_TILE_ORDER_CUH

#include <math.h>
#include <stdint.h>

namespace cocons {

// Tile rasterisation.  Tiles are visited band by band (32 tile rows = 4096 matrix rows per band),
// column by column inside a band, so that the ~300 tiles in flight at any time share one slab of A rows
// (25 MB at K = 768, L2-resident) and a few B column tiles: the operand panel (300 MB at n = 50k, larger than
// L2) is read from HBM once per band instead of once per tile column.  Band height 16 / 24 / 32 run at the
// same speed (35.40 / 35.37 / 35.34 TFLOP/s, tensor-bound); the taller band re-reads the B tiles less often
// (DRAM traffic of the largest launch 1.21x -> ~1.1x algorithmic; profiles/r02_gemm_ncu.md).
//   ni tile rows of 128, njc tile columns of BN = 128 / W; with lower_only, tile (bi, c) exists when
//   bi >= c / W (the matrix origin lies on the diagonal).  Band is the band height in tile rows; the split-int8
//   update numbers super-tiles of 256 rows with Band = kBandRows / 2, so that its bands too are 4096 rows high.
#ifndef COCONS_GEMM_BAND
#define COCONS_GEMM_BAND 32
#endif
constexpr int kBandRows = COCONS_GEMM_BAND;

template <int W, int Band = kBandRows>
__host__ __device__ __forceinline__ int64_t band_tiles(int r, int ni, int njc, int lower_only, int* full_cols_out) {
  const int r0 = r * Band;
  const int h = (ni - r0 < Band) ? ni - r0 : Band;
  if (!lower_only) {
    *full_cols_out = njc;
    return (int64_t)h * njc;
  }
  const int full_cols = (W * r0 < njc) ? W * r0 : njc;  // columns that see all h rows of the band
  *full_cols_out = full_cols;
  int64_t count = (int64_t)h * full_cols;
  const int tri_end = (W * (r0 + h) < njc) ? W * (r0 + h) : njc;
  if (tri_end == W * (r0 + h)) {
    count += (int64_t)W * h * (h + 1) / 2;
  } else {
    for (int c = W * r0; c < tri_end; ++c) count += r0 + h - c / W;
  }
  return count;
}

template <int W, int Band = kBandRows>
__host__ __device__ __forceinline__ int64_t total_tiles(int ni, int njc, int lower_only) {
  int64_t total = 0;
  int dummy;
  for (int r = 0; r * Band < ni; ++r) total += band_tiles<W, Band>(r, ni, njc, lower_only, &dummy);
  return total;
}

// O(1) inverse of the numbering above (a CTA decodes its tile once; a linear walk over the bands
// would cost microseconds for the far-down tiles of a 1500-band-row update).
//   bands [0, rt): complete triangle part      count(r) = W h^2 r + W h (h + 1) / 2   (h = Band)
//   band rt (at most one): triangle clipped by njc or by the last, shorter band - walked directly
//   bands after it: rectangles of h x njc
template <int W, int Band = kBandRows>
__host__ __device__ __forceinline__ void tile_decode(int64_t t, int ni, int njc, int lower_only, int& bi, int& bj) {
  const int nbands = (ni + Band - 1) / Band;
  int r;
  if (!lower_only) {
    r = (int)(t / ((int64_t)Band * njc));
    if (r > nbands - 1) r = nbands - 1;
    t -= (int64_t)r * Band * njc;
    const int r0 = r * Band;
    const int h = (ni - r0 < Band) ? ni - r0 : Band;
    bj = (int)(t / h);
    bi = r0 + (int)(t % h);
    return;
  }
  // number of leading bands that are full height and whose triangle is not clipped by njc
  int rt = njc / (Band * W);
  const int full_height = ni / Band;
  if (rt > full_height) rt = full_height;
  // S(r) = per_a r (r - 1) + per_b r tiles before band r (h = Band: W h^2 r + W h (h + 1) / 2 tiles in band r)
  const int64_t per_a = (int64_t)W * Band * Band / 2, per_b = (int64_t)W * Band * (Band + 1) / 2;
  auto before = [&](int rr) { return per_a * rr * (int64_t)(rr - 1) + per_b * rr; };
  if (t < before(rt)) {
    const double a = (double)per_a, b = (double)(per_b - per_a);
    r = (int)((-b + sqrt(b * b + 4.0 * a * (double)t)) / (2.0 * a));
    if (r < 0) r = 0;
    while (r + 1 <= rt && before(r + 1) <= t) ++r;
    while (before(r) > t) --r;
    t -= before(r);
  } else {
    t -= before(rt);
    r = rt;
    int dummy;
    for (;; ++r) {  // at most two irregular bands, then rectangles in closed form
      const int64_t cnt = band_tiles<W, Band>(r, ni, njc, 1, &dummy);
      if (t < cnt) break;
      t -= cnt;
      const int r0n = (r + 1) * Band;
      if (W * r0n >= njc && ni - r0n >= Band) {  // from here on: full-height rectangles h x njc
        const int64_t rect = (int64_t)Band * njc;
        int skip = (int)(t / rect);
        const int max_skip = (ni - r0n) / Band - 1;  // keep the last (possibly shorter) band for the walk
        if (skip > max_skip) skip = max_skip < 0 ? 0 : max_skip;
        r += skip;
        t -= (int64_t)skip * rect;
      }
    }
  }
  const int r0 = r * Band;
  const int h = (ni - r0 < Band) ? ni - r0 : Band;
  const int full_cols = (W * r0 < njc) ? W * r0 : njc;
  if (t < (int64_t)h * full_cols) {
    bj = (int)(t / h);
    bi = r0 + (int)(t % h);
    return;
  }
  t -= (int64_t)h * full_cols;
  for (int c = W * r0;; ++c) {  // at most W * h columns in the triangular part
    const int rows = r0 + h - c / W;
    if (t < rows) {
      bj = c;
      bi = c / W + (int)t;
      return;
    }
    t -= rows;
  }
}

}  // namespace cocons

#endif
