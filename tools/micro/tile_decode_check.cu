// Exhaustive host check of the trailing-update tile numbering (csrc/chol.cu: total_tiles / tile_decode): for
// every shape the decode must be a bijection onto the expected tile set.  Runs on the CPU (no kernel launched):
//   nvcc -O2 -std=c++17 -gencode arch=compute_100a,code=sm_100a [-DCOCONS_GEMM_BAND=h] tools/micro/tile_decode_check.cu -o tile_decode_check && ./tile_decode_check
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../../cocons_b200/csrc/chol.cu"
namespace cocons { void note_launch(int) {} void set_error(const char*, ...) {} }

template <int W, int Band = cocons::kBandRows>
static long check(int ni, int njc, int lower) {
  const int64_t total = cocons::total_tiles<W, Band>(ni, njc, lower);
  std::vector<unsigned char> seen((size_t)ni * njc, 0);
  long bad = 0;
  int64_t expect = 0;
  for (int bi = 0; bi < ni; ++bi)
    for (int c = 0; c < njc; ++c)
      if (!lower || bi >= c / W) ++expect;
  if (expect != total) return 1 + llabs(expect - total);
  for (int64_t t = 0; t < total; ++t) {
    int bi = -1, bj = -1;
    cocons::tile_decode<W, Band>(t, ni, njc, lower, bi, bj);
    if (bi < 0 || bi >= ni || bj < 0 || bj >= njc || (lower && bi < bj / W) || seen[(size_t)bi * njc + bj]++) ++bad;
  }
  return bad;
}

int main() {
  long shapes = 0, bad = 0;
  for (int ni = 1; ni <= 420; ++ni) {
    const int step = ni < 80 ? 1 : 7;
    for (int nj = 1; nj <= ni; nj += step) {
      bad += check<1>(ni, nj, 1), bad += check<2>(ni, 2 * nj, 1), shapes += 2;
      if (nj <= 12) bad += check<1>(ni, nj, 0), bad += check<2>(ni, 2 * nj, 0), shapes += 2;
    }
    bad += check<2>(ni, 2 * ni, 1), bad += check<1>(ni, ni, 1), shapes += 2;
  }
  for (int ni : {781, 782, 1563, 1564}) bad += check<2>(ni, 2 * ni, 1), bad += check<2>(ni, 12, 1), bad += check<1>(ni, 1, 0), shapes += 3;
  // the super-tiles of the split-int8 update (syrk_i8.cu): 256 x 128 (2 x 2 clusters, the default), 128 x 128 and
  // 256 x 64, bands of 4096 rows; ns super-rows of an update of ni tile rows (odd ni included) and the (a) update
  for (int ni = 1; ni <= 840; ni += (ni < 160 ? 1 : 5)) {
    const int ns = (ni + 1) / 2;
    bad += check<2, cocons::kBandRows / 2>(ns, ni, 1), bad += check<2, cocons::kBandRows / 2>(ns, 6, 1);
    bad += check<1, cocons::kBandRows>(ni, ni, 1), bad += check<4, cocons::kBandRows / 2>(ns, 2 * ni, 1);
    bad += check<2, cocons::kBandRows / 2>(ns, ni, 0), shapes += 5;
  }
  for (int ni : {781, 782, 1563, 1564}) bad += check<2, cocons::kBandRows / 2>((ni + 1) / 2, ni, 1), ++shapes;
  printf("TILE_DECODE band=%d: %ld shapes, %ld wrong\n", cocons::kBandRows, shapes, bad);
  return bad != 0;
}
