"""The super-tile numbering of the split-int8 update (csrc/syrk_i8.cu, clusters of 2 x 2 tiles: 256 rows x one
128-wide block column, bands of 4096 rows): total_tiles / tile_decode of csrc/tile_order.cuh with W = 2 and
Band = 16 must be a bijection onto the super-tiles that hold at least one lower 128 x 64 tile, for odd and even
numbers of tile rows (the missing row of an odd number counted), and for the narrow (a) update.  Compiled for the
host with the system C++ compiler."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SRC = r"""
#define __host__
#define __device__
#define __forceinline__ inline
#include <cstdio>
#include <vector>
#include "tile_order.cuh"
using namespace cocons;

// super-tiles (R, C): 2 tile rows x 2 tile columns of 64; tile (bi, bj) is lower when bi >= bj / 2.  With an odd ni
// the last super-row counts its missing tile row (whose CTAs feed their cluster and store nothing)
static long check(int ni, int nj, int lower) {
  const int ns = (ni + 1) / 2, ncs = nj / 2;
  std::vector<unsigned char> want((size_t)ns * ncs, 0), seen((size_t)ns * ncs, 0);
  long expect = 0, bad = 0;
  for (int R = 0; R < ns; ++R)
    for (int C = 0; C < ncs; ++C) {
      bool any = false;
      for (int bi = 2 * R; bi < 2 * R + 2; ++bi)
        for (int bj = 2 * C; bj < 2 * C + 2; ++bj) any = any || !lower || bi >= bj / 2;
      want[(size_t)R * ncs + C] = any, expect += any;
    }
  const int64_t total = total_tiles<2, kBandRows / 2>(ns, ncs, lower);
  if (total != expect) return 1;
  for (int64_t t = 0; t < total; ++t) {
    int R = -1, C = -1;
    tile_decode<2, kBandRows / 2>(t, ns, ncs, lower, R, C);
    if (R < 0 || R >= ns || C < 0 || C >= ncs || !want[(size_t)R * ncs + C] || seen[(size_t)R * ncs + C]++) ++bad;
  }
  return bad;
}

int main() {
  long shapes = 0, bad = 0;
  for (int ni = 1; ni <= 700; ni += ni < 130 ? 1 : 3) {
    bad += check(ni, 2 * ni, 1) + check(ni, 12, 1) + check(ni, 2 * ni, 0), shapes += 3;
    if (ni >= 6) bad += check(ni, 2 * (ni - 6), 1), ++shapes;  // (b) of an update whose (a) took 6 tile columns
  }
  printf("%ld shapes, %ld wrong\n", shapes, bad);
  return bad != 0;
}
"""


@pytest.mark.skipif(shutil.which("c++") is None, reason="no host C++ compiler")
def test_super_tile_numbering_is_a_bijection(tmp_path):
    src, exe = tmp_path / "check.cpp", tmp_path / "check"
    src.write_text(SRC)
    subprocess.check_call(["c++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "cocons_b200", "csrc"), str(src),
                           "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    print(out.stdout)
    assert out.returncode == 0 and out.stdout.endswith(" 0 wrong\n"), out.stdout + out.stderr
