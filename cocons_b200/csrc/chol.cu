// Blocked right-looking Cholesky on the device (FP64), replacing the LAPACK
// dpotrf behind base::chol at R/neg2loglikelihood.R:136,200,259, R/sim.R:106,162
// and R/optim.R:336.  Lower factor, in place on a column-major matrix padded to
// a multiple of 128 (identity in the padding).
//
//   potrf_tile_kernel   K3: 128x128 diagonal tile, factor + explicit inverse
//   gemm_nt_tma_kernel  K4/K5: C (-)= A B^T on FP64 tensor cores (DMMA.8x8x4 via
//                       mma.sync.m8n8k4.f64), operands streamed global->shared by
//                       the bulk-copy (TMA) engine onto mbarriers; used for the panel
//                       solve (X = A inv(L_jj)^T), the in-panel update and the
//                       trailing SYRK update
//   chol_factor         two-level driver: 128-wide steps inside 512- or 768-wide panels
#include <algorithm>
#include <type_traits>

#include "../../include/cocons_b200.h"
#include "common.cuh"
#include "tile_order.cuh"

namespace cocons {

// ---------------------------------------------------------------------------
// DMMA NT GEMM.  C[M x N] (-)= A[M x K] * B[N x K]^T, everything column-major,
// M, N multiples of 128, K a multiple of 16.
//
// CTA tile 128(i) x 64(j) (128 x 128 for the panel solve), warp tile 32(i) x 32(j).
// The mma's M dimension runs over matrix COLUMNS j and its N dimension over
// matrix ROWS i, so that the two accumulator registers of a thread are two
// consecutive rows of one column; with fragment row g of the tile pair
// (2u, 2u+1) bound to matrix rows {2g, 2g+1} + 16u a thread ends up owning 4
// consecutive rows (32 B) and a quad 128 contiguous bytes of a column.  The
// same binding makes every operand fetch one conflict-free LDS.128.
// ---------------------------------------------------------------------------
#ifndef COCONS_GEMM_RELEASE
#define COCONS_GEMM_RELEASE 1
#endif
constexpr int GBM = 128, GBK = 16, GSTAGES = 4;
constexpr int GLDA = GBM + 4;  // padded leading dimension of a shared k-row (== 4 mod 16: conflict-free LDS.128)
constexpr int kGemmMapped = 2;  // gemm_nt_tma_kernel's tile-mapped C -= A B^T (tiled factor, csrc/capi.cu)

template <int BN, int NU = 2>
struct GemmCfg {
  static constexpr int kWarpI = 16 * NU;             // warp tile is (16 NU)(i) x 32(j); NU = 2: 32 x 32
  static constexpr int kWarpsI = GBM / kWarpI;
  static constexpr int kWarpsJ = BN / 32;
  static constexpr int kThreads = kWarpsI * kWarpsJ * 32;
  static constexpr int kLdb = BN + 4;
  static constexpr int kStageDoubles = GBK * (GLDA + kLdb);
  static constexpr int kSmemBytes = GSTAGES * kStageDoubles * (int)sizeof(double);
  // BN = 64: 8 warps of 32 x 32 (116 registers) and ~100 KB of shared memory per CTA, so TWO CTAs share an
  // SM (4 warps per scheduler): one runs its main loop while the other is in its prologue or its
  // read-modify-write epilogue.  BN = 128 (in-place panel solve): 16 warps, one CTA per SM.
  static constexpr int kMinBlocks = (BN == 64) ? 2 : 1;
};

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(d0), "+d"(d1)
      : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------
// Operand feed: the bulk-copy (TMA) engine.  One elected lane issues, per stage, 32 `cp.async.bulk` row
// copies (16 k-rows of A and of B, each a contiguous 1 KB / BN*8 B segment of a matrix column) straight
// into the padded shared rows; the bytes land on an mbarrier (`complete_tx`).  Consumers wait on that
// barrier and hand the slot back through an `empty` mbarrier - no __syncthreads, no per-thread address
// arithmetic in the MMA warps.  The producer role rotates over the warps (stage s is issued by warp
// s mod nwarps) so that no warp is permanently behind.  One tile per CTA.
// (An earlier version fed the operands with per-thread cp.async/LDGSTS and a block barrier per stage:
// 31.9 TFLOP/s against 35.3 for this one; the ablation is in profiles/r01_gemm_tma_v3_ncu.md.)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive whose barrier address depends on x and y (zero is 0 at run time, unknown at compile time): the
// instruction cannot issue before the instructions that produce x and y have completed
__device__ __forceinline__ void mbar_arrive_after(uint32_t bar, double x, double y, uint32_t zero) {
  asm volatile(
      "{\n"
      ".reg .b32 xl, xh, yl, yh;\n"
      "mov.b64 {xl, xh}, %1;\n"
      "mov.b64 {yl, yh}, %2;\n"
      "or.b32 xl, xl, yl;\n"
      "and.b32 xl, xl, %3;\n"
      "add.u32 xl, xl, %0;\n"
      "mbarrier.arrive.shared::cta.b64 _, [xl];\n"
      "}" ::"r"(bar),
      "d"(x), "d"(y), "r"(zero)
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// ASSIGN 0: C -= A B^T; 1: C = A B^T; 2 (kGemmMapped): C -= A B^T with every 128 x 128 block of C looked up in a
// tile map, so that one launch updates tiles scattered over the panels of a tiled factor.  In that mode `ldc`
// carries the device address of the map, int64: [pairs: element offset of the target block from C][128-column
// blocks: leading dimension of the target], pair (bi, c) numbered bi (bi + 1) / 2 + c with lower_only, bi * nj / 2 + c
// without (c = the 128-column block of the CTA's tile).
template <int BN, int NU, int ASSIGN>
__global__ void __launch_bounds__(GemmCfg<BN, NU>::kThreads, GemmCfg<BN, NU>::kMinBlocks)
    gemm_nt_tma_kernel(int ni, int nj, int64_t K, const double* A, int64_t lda, const double* B, int64_t ldb,
                       double* C, int64_t ldc, int lower_only) {
  using Cfg = GemmCfg<BN, NU>;
  constexpr int kWarps = Cfg::kThreads / 32;
  constexpr uint32_t kStageBytes = GBK * (GBM + BN) * (uint32_t)sizeof(double);
  extern __shared__ __align__(16) double smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)GSTAGES * Cfg::kStageDoubles);
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, c4 = lane & 3;
  const int iw = (warp % Cfg::kWarpsI) * Cfg::kWarpI, jw = (warp / Cfg::kWarpsI) * 32;
  int bi, bj;
  tile_decode<GBM / BN>(blockIdx.x, ni, nj, lower_only, bi, bj);
  const double* Ag = A + (int64_t)bi * GBM;
  const double* Bg = B + (int64_t)bj * BN;
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + GSTAGES);
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < GSTAGES; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, kWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  const int64_t nkb = K / GBK;
  const uint32_t stage0 = smem_u32(smem);
  const uint32_t rt_zero = (uint32_t)((uint64_t)lda >> 48);  // 0 for any real leading dimension; not foldable
  (void)rt_zero;
  auto produce = [&](int64_t ld) {  // one lane
    const int slot = (int)(ld % GSTAGES);
    const int64_t fill = ld / GSTAGES;
    if (fill >= 1) mbar_wait(empty0 + 8 * slot, (uint32_t)((fill - 1) & 1));
    const uint32_t fb = full0 + 8 * slot;
    mbar_expect_tx(fb, kStageBytes);
    const uint32_t da = stage0 + (uint32_t)slot * Cfg::kStageDoubles * 8u;
    const uint32_t db = da + GBK * GLDA * 8u;
    const double* a = Ag + ld * GBK * lda;
    const double* b = Bg + ld * GBK * ldb;
#pragma unroll
    for (int k = 0; k < GBK; ++k) bulk_g2s(da + k * GLDA * 8u, a + (int64_t)k * lda, GBM * 8u, fb);
#pragma unroll
    for (int k = 0; k < GBK; ++k) bulk_g2s(db + k * Cfg::kLdb * 8u, b + (int64_t)k * ldb, BN * 8u, fb);
  };

  double acc[4][2 * NU][2];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 2 * NU; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;

  if (ASSIGN == kGemmMapped) {  // C and ldc of the target block (BN = 64: two CTA tiles per 128-column block)
    static_assert(ASSIGN != kGemmMapped || BN == 64, "the tile map is for 128 x 64 CTA tiles");
    const int64_t* map = reinterpret_cast<const int64_t*>(ldc);
    const int c = bj / 2;
    const int64_t pair = lower_only ? (int64_t)bi * (bi + 1) / 2 + c : (int64_t)bi * (nj / 2) + c;
    const int64_t npairs = lower_only ? (int64_t)ni * (ni + 1) / 2 : (int64_t)ni * (nj / 2);
    ldc = map[npairs + c];
    // shifted so that the addressing below, C + bj BN ldc + bi GBM, lands on the target block
    C += map[pair] + (int64_t)(bj & 1) * BN * ldc - (int64_t)bj * BN * ldc - (int64_t)bi * GBM;
  }
#ifndef COCONS_GEMM_NO_PREFETCH
  if (ASSIGN != 1) {  // pull the C tile towards L2 while the main loop runs
    const double* Cp = C + (int64_t)bj * BN * ldc + (int64_t)bi * GBM;
    for (int l = tid; l < BN * 8; l += Cfg::kThreads)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(Cp + (int64_t)(l >> 3) * ldc + (l & 7) * 16));
  }
#endif
  if (warp == 0 && lane == 0)
    for (int s = 0; s < GSTAGES - 1 && s < nkb; ++s) produce(s);
  __syncwarp();

  for (int64_t it = 0; it < nkb; ++it) {
    const int64_t ld = it + GSTAGES - 1;
    if (ld < nkb && warp == (int)(it % kWarps) && lane == 0) produce(ld);
    __syncwarp();
    const int slot = (int)(it % GSTAGES);
    mbar_wait(full0 + 8 * slot, (uint32_t)((it / GSTAGES) & 1));
    const double* as = smem + (size_t)slot * Cfg::kStageDoubles + iw + 2 * g;
    const double* bs = smem + (size_t)slot * Cfg::kStageDoubles + GBK * GLDA + jw + 2 * g;
#pragma unroll
    for (int kk = 0; kk < GBK / 4; ++kk) {
      const int k = kk * 4 + c4;
      double fi[2 * NU], fj[4];
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        const double2 v = *reinterpret_cast<const double2*>(as + k * GLDA + 16 * u);
        fi[2 * u] = v.x;
        fi[2 * u + 1] = v.y;
      }
#pragma unroll
      for (int v2 = 0; v2 < 2; ++v2) {
        const double2 v = *reinterpret_cast<const double2*>(bs + k * Cfg::kLdb + 16 * v2);
        fj[2 * v2] = v.x;
        fj[2 * v2 + 1] = v.y;
      }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 2 * NU; ++b) dmma884(acc[a][b][0], acc[a][b][1], fj[a], fi[b]);
    }
    // Handing the slot back.  The next fill is written by the bulk-copy engine (async proxy) while this
    // warp read the slot with ordinary LDS (generic proxy): a write-after-read across proxies.  ptxas
    // places SYNCS.ARRIVE right behind the ISSUE of the last LDS - ahead of the DMMAs that consume the
    // loaded registers - and the arrive does not wait for the load unit: with the LSU queue backed up
    // (the co-resident CTA's epilogue), the producer saw the slot free, refilled it, and a late LDS read
    // a 128-byte piece of the NEXT k-block (round 1's irreproducible factors, profiles/r02_chol_race.md).
    //   COCONS_GEMM_RELEASE bit 0: fence.proxy.async.shared::cta before the arrive (the documented
    //     generic->async ordering, same place as CUTLASS's fence_view_async_shared() before consumer_release)
    //   bit 1: the arrive's address is made data-dependent on two accumulators that between them consume
    //     every LDS of the stage, so it cannot issue before those loads have delivered
    __syncwarp();
#if (COCONS_GEMM_RELEASE & 1)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
#endif
#if (COCONS_GEMM_RELEASE & 2)
    if (lane == 0) mbar_arrive_after(empty0 + 8 * slot, acc[0][2][0], acc[2][0][0], rt_zero);
#else
    if (lane == 0) mbar_arrive(empty0 + 8 * slot);
#endif
  }

  double* Cg = C + (int64_t)bj * BN * ldc + (int64_t)bi * GBM;
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int j = jw + 16 * (a >> 1) + 2 * g + (a & 1);
#pragma unroll
    for (int u = 0; u < NU; ++u) {
      const int r0 = iw + 16 * u + 4 * c4;
      double2* p = reinterpret_cast<double2*>(Cg + (int64_t)j * ldc + r0);
      double2 lo, hi;
      if (ASSIGN == 1) {
        lo.x = acc[a][2 * u][0];
        lo.y = acc[a][2 * u + 1][0];
        hi.x = acc[a][2 * u][1];
        hi.y = acc[a][2 * u + 1][1];
      } else {
        // C is touched once per launch: streaming loads and stores (evict-first), so that the 19 GB of C going
        // through L2 do not push out the A slab and the B tiles that the other CTAs of the band re-use
        lo = __ldcs(p);
        hi = __ldcs(p + 1);
        lo.x -= acc[a][2 * u][0];
        lo.y -= acc[a][2 * u + 1][0];
        hi.x -= acc[a][2 * u][1];
        hi.y -= acc[a][2 * u + 1][1];
      }
      if (ASSIGN == 1) {
        p[0] = lo;
        p[1] = hi;
      } else {
        __stcs(p, lo);
        __stcs(p + 1, hi);
      }
    }
  }
}

// mode 0: C -= A B^T on 128 x 64 tiles, 8 warps, two CTAs per SM; mode 1: C = A B^T on 128 x 128 tiles,
// 16 warps, one CTA per SM - the in-place panel solve needs one CTA to own the whole 128-column block
// it overwrites (every bulk copy of its A rows has landed before its first store).
// COCONS_DEBUG_SYNC=1: host-synchronise the stream before every GEMM launch (bisection aid, see DESIGN.md §4a)
static int debug_sync_mode() {
  static int m = -1;
  if (m < 0) m = getenv("COCONS_DEBUG_SYNC") ? 1 : 0;
  return m;
}

// 128 x 64 tiles: C -= A B^T (EPI = 0) or the tile-mapped variant (EPI = kGemmMapped)
template <int EPI>
static void launch_gemm_64(int ni, int nj, int64_t K, const double* A, int64_t lda, const double* B, int64_t ldb,
                           double* C, int64_t ldc, int lower_only, cudaStream_t st) {
  const int64_t tiles = total_tiles<2>(ni, nj, lower_only);
  gemm_nt_tma_kernel<64, 2, EPI><<<(unsigned)tiles, GemmCfg<64, 2>::kThreads, GemmCfg<64, 2>::kSmemBytes + 64, st>>>(
      ni, nj, K, A, lda, B, ldb, C, ldc, lower_only);
}

// mode 2: as mode 0 with C addressed through a tile map whose device address is passed as ldc (see the kernel)
void launch_gemm_nt(int mode, int64_t M, int64_t N, int64_t K, const double* A, int64_t lda, const double* B,
                    int64_t ldb, double* C, int64_t ldc, int lower_only, cudaStream_t st) {
  if (M <= 0 || N <= 0 || K <= 0) return;
  static bool attr_done[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (debug_sync_mode()) cudaStreamSynchronize(st);
  if (dev < 16 && !attr_done[dev]) {
    cudaFuncSetAttribute(gemm_nt_tma_kernel<64, 2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         GemmCfg<64, 2>::kSmemBytes + 64);
    cudaFuncSetAttribute(gemm_nt_tma_kernel<128, 2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         GemmCfg<128, 2>::kSmemBytes + 64);
    cudaFuncSetAttribute(gemm_nt_tma_kernel<64, 2, kGemmMapped>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         GemmCfg<64, 2>::kSmemBytes + 64);
    attr_done[dev] = true;
  }
  const int ni = (int)(M / GBM);
  note_launch();
  if (mode == 1) {
    const int nj = (int)(N / 128);
    const int64_t tiles = total_tiles<1>(ni, nj, lower_only);
    gemm_nt_tma_kernel<128, 2, 1><<<(unsigned)tiles, GemmCfg<128, 2>::kThreads, GemmCfg<128, 2>::kSmemBytes + 64, st>>>(
        ni, nj, K, A, lda, B, ldb, C, ldc, lower_only);
  } else if (mode == kGemmMapped) {
    launch_gemm_64<kGemmMapped>(ni, (int)(N / 64), K, A, lda, B, ldb, C, ldc, lower_only, st);
  } else {
    launch_gemm_64<0>(ni, (int)(N / 64), K, A, lda, B, ldb, C, ldc, lower_only, st);
  }
}

// ---------------------------------------------------------------------------
// Diagonal tile: Cholesky of a 128 x 128 tile and, in the SAME sweep, its explicit inverse
// W = L^-1 (which turns the panel solve and the later forward substitutions into plain
// products), with both matrices held in REGISTERS.
//
// 256 threads as a 16 x 16 grid, thread (tx, ty) = (tid >> 4, tid & 15) owns the 2-D cyclic set
// (i = ty + 16 a, j = tx + 16 b), a >= b, of L and of W.  Step k applies, to registers,
//     L[i][j] -= L[i][k] L[j][k]                        (right-looking Cholesky)
//     W[i][c] -= L[i][k] / L[k][k] * W~[k][c]            (forward elimination of the identity)
// after column k of L (scaled by rsqrt(pivot), pivot broadcast by half-warp shuffle) and the still
// unscaled row k of W have been published in 1 KB shared vectors.
//
// The column is the critical path, so it runs one step AHEAD: inside step k every thread first
// updates only what step k+1 publishes (column k+1 of L, row k+1 of W), the owners publish it and
// everybody ARRIVES on the mbarrier of step k+1, and only then is the bulk of step k's update done -
// the next pivot / rsqrt / scale overlaps the other warps' FMAs.  Three buffers and three mbarriers
// (k mod 3) make that safe: a buffer is rewritten two steps after its last reader started.
// ---------------------------------------------------------------------------
constexpr int PT = kTile;
#ifdef COCONS_POTRF_PROBE
__device__ long long g_probe[PT * 8];
#define PROBE(slot, kk, cond) if (cond) g_probe[(kk) * 8 + (slot)] = clock64()
#else
#define PROBE(slot, kk, cond)
#endif

__global__ void __launch_bounds__(256, 1)
    potrf_tile_kernel(double* __restrict__ A, int64_t ld, double* __restrict__ Winv, int* __restrict__ info,
                      int first_index) {
  __shared__ double colbuf[3][PT];
  __shared__ double rowbuf[3][PT];
  __shared__ double rdiag[3];
  __shared__ __align__(8) uint64_t mbar[3];
  __shared__ int fail;
  const int tid = threadIdx.x, lane = tid & 31;
  const int tx = tid >> 4, ty = tid & 15;
  const unsigned hmask = 0xFFFFu << (lane & 16);
  double r[8][8], w[8][8];
#pragma unroll
  for (int b = 0; b < 8; ++b)
#pragma unroll
    for (int a = 0; a < 8; ++a) {
      w[a][b] = 0.0;
      r[a][b] = (a >= b) ? __ldcv(A + (int64_t)(tx + 16 * b) * ld + ty + 16 * a) : 0.0;
    }
  if (tid == 0) {
    fail = 0;
    for (int m = 0; m < 3; ++m) mbar_init(smem_u32(&mbar[m]), 256);
  }
  __syncthreads();

  // publish column `kk` of L (its owners: tx == kk % 16) and row `kk` of W (ty == kk % 16); NB = kk / 16
  auto publish = [&](auto nb_tag, int kk) {
    constexpr int NB = decltype(nb_tag)::value;
    const int qx = kk & 15;
    double* cb = colbuf[kk % 3];
    double* rb = rowbuf[kk % 3];
    if (tx == qx) {
      PROBE(1, kk, ty == qx);
      const double d = __shfl_sync(hmask, r[NB][NB], (lane & 16) | qx);
      PROBE(2, kk, ty == qx);
      // one reciprocal square root on the critical path (dpotf2 scales by 1/sqrt(d) as well)
      const double rinv = rsqrt(d), piv = d * rinv;
      PROBE(3, kk, ty == qx && rinv > 0);
#pragma unroll
      for (int a = 0; a < 8; ++a) {  // rows above block NB are never read by the consumers of this column
        const int i = ty + 16 * a;
        if (a >= NB) {
          double v = r[a][NB];
          v = (i > kk) ? v * rinv : ((i == kk) ? piv : v);
          r[a][NB] = v;
          cb[i] = (i > kk) ? v : 0.0;
        }
      }
      if (ty == qx) {
        rdiag[kk % 3] = rinv;
        if (!(d > 0.0)) {  // non-positive or NaN pivot: dpotrf's info = k+1
          fail = 1;
          atomicCAS(info, 0, first_index + kk + 1);
        }
      }
    }
    if (ty == qx) {  // row kk of W, unscaled, 1 on the diagonal, 0 right of it (blocks right of NB are
                     // never read by the consumers of this row)
#pragma unroll
      for (int b = 0; b < 8; ++b) {
        const int c = tx + 16 * b;
        if (b <= NB) rb[c] = (c < kk) ? w[NB][b] : ((c == kk) ? 1.0 : 0.0);
      }
    }
    PROBE(4, kk, tx == qx && ty == qx);
    mbar_arrive(smem_u32(&mbar[kk % 3]));
    PROBE(5, kk, tx == qx && ty == qx);
  };

  publish(std::integral_constant<int, 0>{}, 0);

  bool stop = false;
  auto block_steps = [&](auto kb_tag) {  // the 16 steps of block column kb (kb is a compile-time index)
    constexpr int kb = decltype(kb_tag)::value;
#pragma unroll 1
    for (int kx = 0; kx < 16 && !stop; ++kx) {
      const int k = kb * 16 + kx;
      mbar_wait(smem_u32(&mbar[k % 3]), (uint32_t)((k / 3) & 1));
      PROBE(0, k + 1, tx == ((k + 1) & 15) && ty == ((k + 1) & 15));
      PROBE(6, k, tid == 255);
      stop = (*(volatile int*)&fail != 0);
      if (stop) break;
      const double* cb = colbuf[k % 3];
      const double* rb = rowbuf[k % 3];
      const double rinv = rdiag[k % 3];
      double li[8], lw[8];
#pragma unroll
      for (int a = 0; a < 8; ++a) {
        li[a] = (a >= kb) ? cb[ty + 16 * a] : 0.0;  // zero for i <= k
        lw[a] = li[a] * rinv;
      }
      // the update of step k, restricted to block column PB of L and block row PB of W (ONLY = true)
      // or to everything else (ONLY = false)
      auto update = [&](auto pb_tag, auto only_tag) {
        constexpr int PB = decltype(pb_tag)::value;
        constexpr bool ONLY = decltype(only_tag)::value;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          if (b >= kb && ((b == PB) == ONLY)) {
            const double lj = cb[tx + 16 * b];  // zero for j <= k: finished columns stay untouched
#pragma unroll
            for (int a = 0; a < 8; ++a)
              if (a >= b) r[a][b] = fma(-li[a], lj, r[a][b]);
          }
          if (b <= kb) {
            const double wk = rb[tx + 16 * b];  // row k of W before its scaling, zero right of column k
#pragma unroll
            for (int a = 0; a < 8; ++a)
              if (a >= kb && a >= b && ((a == PB) == ONLY)) w[a][b] = fma(-lw[a], wk, w[a][b]);
          }
        }
      };
      if (k + 1 < PT) {
        if (kx < 15) {  // step k+1 lives in the same 16-block
          update(std::integral_constant<int, kb>{}, std::true_type{});
          publish(std::integral_constant<int, kb>{}, k + 1);
          update(std::integral_constant<int, kb>{}, std::false_type{});
        } else {
          constexpr int NB = (kb < 7) ? kb + 1 : 7;
          update(std::integral_constant<int, NB>{}, std::true_type{});
          publish(std::integral_constant<int, NB>{}, k + 1);
          update(std::integral_constant<int, NB>{}, std::false_type{});
        }
      } else {
        update(std::integral_constant<int, 99>{}, std::false_type{});
      }
      PROBE(7, k, tid == 255);
      if (ty == kx) {  // row k of W is final once scaled (its own update above was a no-op: li = 0 there)
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          const int c = tx + 16 * b;
          if (b <= kb) w[kb][b] = (c < k) ? w[kb][b] * rinv : ((c == k) ? rinv : w[kb][b]);
        }
      }
    }
  };
  block_steps(std::integral_constant<int, 0>{});
  block_steps(std::integral_constant<int, 1>{});
  block_steps(std::integral_constant<int, 2>{});
  block_steps(std::integral_constant<int, 3>{});
  block_steps(std::integral_constant<int, 4>{});
  block_steps(std::integral_constant<int, 5>{});
  block_steps(std::integral_constant<int, 6>{});
  block_steps(std::integral_constant<int, 7>{});
  if (stop) return;

  // L back to the matrix (the strict upper part of the tile is zeroed) and W = L^-1, 128 x 128
  // column-major, zero above the diagonal
#pragma unroll
  for (int b = 0; b < 8; ++b)
#pragma unroll
    for (int a = 0; a < 8; ++a) {
      const int i = ty + 16 * a, j = tx + 16 * b;
      const bool low = (a >= b && i >= j);
      A[(int64_t)j * ld + i] = low ? r[a][b] : 0.0;
      Winv[j * PT + i] = low ? w[a][b] : 0.0;
    }
}

// ---------------------------------------------------------------------------
// Diagonal tile, blocked variant (K3b).  The register-resident kernel above spends ~1000 clocks on each
// of its 128 column steps (pivot -> rsqrt -> publish -> mbarrier round trip); this one shortens the
// sequential part to what is inherently sequential - the 16 pivots of a 16 x 16 diagonal block, done by
// ONE warp - and moves everything else into 16 x 16 x 16 block products on the FP64 tensor cores
// (DMMA.8x8x4), spread over the 8 warps.  The tile and the running inverse live in shared memory as
// 36 + 36 lower blocks of 16 x 16, column-major with a column stride of 20 doubles (every DMMA fragment
// fetch and the coalesced tile load / store are bank-conflict free).
//
// Block step s = 0..7, with T the forward-eliminated identity (T = I at the start):
//   P1 (warp 0)   L_ss = chol(A_ss),  W_ss = L_ss^-1                (16 sequential pivots)
//   P2 (8 warps)  L_as = A_as W_ss^T            a > s               W_sc = W_ss T_sc        c < s
//   P3 (8 warps)  A_ab -= L_as L_bs^T    s < b <= a                 T_ac -= L_as W_sc    a > s, c <= s
// after which W = L^-1.  Same outputs as potrf_tile_kernel: L over the tile (strict upper part zeroed),
// W as a 128 x 128 column-major matrix, first failing pivot (1-based, dpotrf's info) in *info.
// ---------------------------------------------------------------------------
constexpr int PB = 16;                        // block edge
constexpr int PNB = PT / PB;                  // 8 block rows
constexpr int PBS = 20;                       // column stride of a block in shared memory (== 4 mod 16)
constexpr int PBLK = PB * PBS;                // doubles per block
constexpr int PNBLK = PNB * (PNB + 1) / 2;    // 36 lower blocks
constexpr int kPotrfBlockedSmem = 2 * PNBLK * PBLK * (int)sizeof(double) + 16;
#ifdef COCONS_POTRF_PROBE
__device__ long long g_probe_b[64];
#define PROBEB(slot) if (threadIdx.x == 0) g_probe_b[slot] = clock64()
#else
#define PROBEB(slot)
#endif

__device__ __forceinline__ int pblk(int a, int b) { return (a * (a + 1) / 2 + b) * PBLK; }  // a >= b

// Blocks are stored COLUMN-major in shared memory: element (i, j) of a block at [i + j PBS].
//
// One warp: C (16 x 16) = X Y (MODE 0) or C -= X Y (MODE 1), X(i,k) at X[i sxi + k sxk], Y(k,j) at
// Y[k syk + j syj].  Every operand fragment is fetched before the first store, so C may alias X or Y.
// The product is formed transposed (D' = Y^T X^T) so that the two accumulators of a lane are two
// consecutive ROWS of one column of C - contiguous in the column-major block.  mma.m8n8k4.f64 fragments:
// a = A[g][c4], b = B[c4][g], d = D[g][2 c4 + {0,1}]; here A = Y^T (m = column of C), B = X^T (n = row of C).
// A dependent DMMA chain costs ~200 clocks per link, so the 16 products of a block go to 16 independent
// accumulator pairs and are summed afterwards.
template <int MODE>
__device__ __forceinline__ void bmm16(double* C, const double* X, int sxi, int sxk, const double* Y, int syk, int syj,
                                      int lane) {
  const int g = lane >> 2, c4 = lane & 3;
  double xb[2][4], ya[2][4];
#pragma unroll
  for (int q = 0; q < 2; ++q)
#pragma unroll
    for (int kc = 0; kc < 4; ++kc) {
      xb[q][kc] = X[(8 * q + g) * sxi + (4 * kc + c4) * sxk];
      ya[q][kc] = Y[(4 * kc + c4) * syk + (8 * q + g) * syj];
    }
  __syncwarp();
  double d[2][2][4][2];
#pragma unroll
  for (int qi = 0; qi < 2; ++qi)
#pragma unroll
    for (int qj = 0; qj < 2; ++qj)
#pragma unroll
      for (int kc = 0; kc < 4; ++kc) {
        d[qi][qj][kc][0] = d[qi][qj][kc][1] = 0.0;
        // D'[m = g -> column 8 qj + g][n = 2 c4 + {0,1} -> row 8 qi + 2 c4 + {0,1}]
        dmma884(d[qi][qj][kc][0], d[qi][qj][kc][1], ya[qj][kc], xb[qi][kc]);
      }
#pragma unroll
  for (int qi = 0; qi < 2; ++qi)
#pragma unroll
    for (int qj = 0; qj < 2; ++qj) {
      const double s0 = (d[qi][qj][0][0] + d[qi][qj][1][0]) + (d[qi][qj][2][0] + d[qi][qj][3][0]);
      const double s1 = (d[qi][qj][0][1] + d[qi][qj][1][1]) + (d[qi][qj][2][1] + d[qi][qj][3][1]);
      double2* p = reinterpret_cast<double2*>(C + (8 * qj + g) * PBS + 8 * qi + 2 * c4);
      double2 v;
      if (MODE) {
        v = *p;
        v.x -= s0;
        v.y -= s1;
      } else {
        v.x = s0;
        v.y = s1;
      }
      *p = v;
    }
}

// P1 of block step s, one warp: L_ss = chol(A_ss) in place, then W_ss = L_ss^-1 in place of the identity
// block.  Lane j < 16 owns COLUMN j in registers.  Pivot step k: lane k takes the reciprocal square root
// of its diagonal entry, scales its column and stores it - that IS column k of L_ss in the block - then
// every lane j > k pulls l_jk and the broadcast l_ik from there: one __syncwarp per pivot, no shuffles.
// The inverse follows by forward substitution on the columns of the identity (an FMA chain of depth 16).
__device__ __forceinline__ void potrf_diag_block(double* Dl, double* Dt, double* rinvs, int lane, int* fail,
                                                 int* info, int first_pivot) {
  const int j = lane & 15;
  const bool active = lane < 16;
  double v[PB];
#pragma unroll
  for (int i = 0; i < PB; i += 2) {
    const double2 x = *reinterpret_cast<const double2*>(Dl + j * PBS + i);
    v[i] = x.x;
    v[i + 1] = x.y;
  }
#pragma unroll
  for (int k = 0; k < PB; ++k) {
    if (active && j == k) {
      const double d = v[k];
      if (!(d > 0.0) && atomicCAS(fail, 0, 1) == 0) atomicCAS(info, 0, first_pivot + k + 1);  // dpotrf's info
      const double rinv = rsqrt(d);  // (a float-seeded Newton variant measured slower: 305 vs ~160 clocks)
      rinvs[k] = rinv;
      v[k] = d * rinv;
#pragma unroll
      for (int i = k + 1; i < PB; ++i) v[i] *= rinv;
#pragma unroll
      for (int i = 0; i < PB; i += 2) {  // column k of L_ss (rows above k are never read)
        double2 x;
        x.x = v[i];
        x.y = v[i + 1];
        *reinterpret_cast<double2*>(Dl + k * PBS + i) = x;
      }
    }
    __syncwarp();
    if (active && j > k) {
      const double ljk = Dl[k * PBS + j];
#pragma unroll
      for (int i = k + 1; i < PB; ++i)
        if (i >= j) v[i] = fma(-Dl[k * PBS + i], ljk, v[i]);
    }
  }
  // W_ss: lane c owns column c of the eliminated identity; t[k] is final when step k starts
  if (active) {
    double t[PB];
#pragma unroll
    for (int i = 0; i < PB; ++i) t[i] = (i == j) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 0; k < PB - 1; ++k) {
      const double tk = t[k] * rinvs[k];  // zero while k < column
#pragma unroll
      for (int i = k + 1; i < PB; ++i) t[i] = fma(-Dl[k * PBS + i], tk, t[i]);
    }
#pragma unroll
    for (int i = 0; i < PB; i += 2) {
      double2 x;
      x.x = t[i] * rinvs[i];
      x.y = t[i + 1] * rinvs[i + 1];
      *reinterpret_cast<double2*>(Dt + j * PBS + i) = x;
    }
  }
}

__global__ void __launch_bounds__(256, 1)
    potrf_tile_blocked_kernel(double* __restrict__ A, int64_t ld, double* __restrict__ Winv, int* __restrict__ info,
                              int first_index) {
  extern __shared__ __align__(16) double psm[];
  double* Lb = psm;                  // lower blocks of the tile -> L
  double* Tb = psm + PNBLK * PBLK;   // lower blocks of T -> W
  __shared__ int fail;
  __shared__ double rinvs[PB];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) fail = 0;
  PROBEB(0);
  // load: column-major sweep of the tile (coalesced 16-byte loads), lower blocks only; T = 0 off the
  // diagonal blocks (the diagonal blocks of T are written by P1)
#pragma unroll 8
  for (int idx = tid; idx < PT * PT / 2; idx += 256) {
    const int i = (2 * idx) & (PT - 1), j = (2 * idx) >> 7;
    const int a = i >> 4, b = j >> 4;
    if (a >= b) {
      const double2 x = __ldcv(reinterpret_cast<const double2*>(A + (int64_t)j * ld + i));
      const int off = pblk(a, b) + (j & 15) * PBS + (i & 15);
      *reinterpret_cast<double2*>(Lb + off) = x;
      *reinterpret_cast<double2*>(Tb + off) = make_double2(0.0, 0.0);
    }
  }
  __syncthreads();
  PROBEB(1);

  // s = -1 is the prologue (P1 of block 0 only); the diagonal-block routine has ONE call site so that its
  // fully unrolled code is fetched into the instruction cache once
  for (int s = -1; s < PNB; ++s) {
    if (s >= 0) {
      PROBEB(2 + 3 * s);
      if (fail) return;
      double* Dt = Tb + pblk(s, s);  // W_ss
      // ---- P2: panel blocks L_as = A_as W_ss^T (a > s) and the new block row of W, W_sc = W_ss T_sc (c < s)
      int t = 0;
      for (int a = s + 1; a < PNB; ++a, ++t)
        if ((t & 7) == warp) bmm16<0>(Lb + pblk(a, s), Lb + pblk(a, s), 1, PBS, Dt, PBS, 1, lane);
      for (int c = 0; c < s; ++c, ++t)
        if ((t & 7) == warp) bmm16<0>(Tb + pblk(s, c), Dt, 1, PBS, Tb + pblk(s, c), 1, PBS, lane);
      __syncthreads();
      PROBEB(3 + 3 * s);
    }
    // ---- P3: trailing update A_ab -= L_as L_bs^T (s < b <= a) and T_ac -= L_as W_sc (a > s, c <= s).
    // Look-ahead: warp 0 updates only the next diagonal block and factors it (P1 of step s + 1) while the
    // other seven warps do the rest.
    if (warp == 0) {
      if (s + 1 < PNB) {
        if (s >= 0) {
          bmm16<1>(Lb + pblk(s + 1, s + 1), Lb + pblk(s + 1, s), 1, PBS, Lb + pblk(s + 1, s), PBS, 1, lane);
          __syncwarp();
        }
        potrf_diag_block(Lb + pblk(s + 1, s + 1), Tb + pblk(s + 1, s + 1), rinvs, lane, &fail, info,
                         first_index + (s + 1) * PB);
      }
    } else if (s >= 0) {
      int t = 0;
      for (int a = s + 1; a < PNB; ++a) {
        for (int b = s + 1; b <= a; ++b) {
          if (a == s + 1 && b == s + 1) continue;  // warp 0's block
          if (t++ % 7 == warp - 1)
            bmm16<1>(Lb + pblk(a, b), Lb + pblk(a, s), 1, PBS, Lb + pblk(b, s), PBS, 1, lane);
        }
        for (int c = 0; c <= s; ++c)
          if (t++ % 7 == warp - 1)
            bmm16<1>(Tb + pblk(a, c), Lb + pblk(a, s), 1, PBS, Tb + pblk(s, c), 1, PBS, lane);
      }
    }
    __syncthreads();
    if (s >= 0) PROBEB(4 + 3 * s);
  }

  // store: L over the tile (strict upper part zeroed), W = L^-1 column-major, zero above the diagonal
#pragma unroll 4
  for (int idx = tid; idx < PT * PT / 2; idx += 256) {
    const int i = (2 * idx) & (PT - 1), j = (2 * idx) >> 7;
    const int a = i >> 4, b = j >> 4;
    double2 l, w;
    l.x = l.y = w.x = w.y = 0.0;
    if (a >= b) {
      const int off = pblk(a, b) + (j & 15) * PBS + (i & 15);
      const double2 lv = *reinterpret_cast<const double2*>(Lb + off);
      const double2 wv = *reinterpret_cast<const double2*>(Tb + off);
      if (i >= j) l.x = lv.x, w.x = wv.x;
      if (i + 1 >= j) l.y = lv.y, w.y = wv.y;
    }
    *reinterpret_cast<double2*>(A + (int64_t)j * ld + i) = l;
    *reinterpret_cast<double2*>(Winv + j * PT + i) = w;
  }
  PROBEB(30);
}

// the blocked kernel is the default (53.8 vs 81.0 us per cold tile in tools/micro/potrf_check.cu);
// COCONS_POTRF=1 selects the register-resident column-sweep kernel
void launch_potrf_tile(double* A, int64_t ld, double* Winv, int* info, int first_index, cudaStream_t st) {
  static int variant = -1;
  static bool attr_done[16] = {};
  if (variant < 0) {
    const char* e = getenv("COCONS_POTRF");
    variant = e ? atoi(e) : 2;
  }
  note_launch();
  if (variant == 1) {
    potrf_tile_kernel<<<1, 256, 0, st>>>(A, ld, Winv, info, first_index);
    return;
  }
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 16 && !attr_done[dev]) {
    cudaFuncSetAttribute(potrf_tile_blocked_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPotrfBlockedSmem);
    attr_done[dev] = true;
  }
  potrf_tile_blocked_kernel<<<1, 256, kPotrfBlockedSmem, st>>>(A, ld, Winv, info, first_index);
}

SyrkI8Ops g_syrk_i8 = {nullptr, nullptr};

int chol_workspace_create(int64_t n_pad, CholWorkspace* ws, bool with_i8) {
  ws->winv = nullptr, ws->info = nullptr, ws->panel_stream = nullptr, ws->ev_a = nullptr, ws->ev_p = nullptr;
  ws->ev_k0 = nullptr, ws->ev_k1 = nullptr;
  ws->i8_slices = nullptr, ws->i8_scale = nullptr;
  int lo = 0, hi = 0;
  cudaDeviceGetStreamPriorityRange(&lo, &hi);  // hi = greatest priority (numerically lowest)
  if (const char* e = getenv("COCONS_PANEL_PRIORITY"))  // 0: panel stream at default priority (bisection aid)
    if (atoi(e) == 0) hi = 0;
  if (cudaMalloc(&ws->winv, sizeof(double) * (n_pad / kTile) * kTile * kTile) != cudaSuccess ||
      cudaMalloc(&ws->info, sizeof(int)) != cudaSuccess ||
      cudaStreamCreateWithPriority(&ws->panel_stream, cudaStreamNonBlocking, hi) != cudaSuccess ||
      cudaEventCreateWithFlags(&ws->ev_a, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ws->ev_p, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&ws->ev_k0) != cudaSuccess || cudaEventCreate(&ws->ev_k1) != cudaSuccess) {
    chol_workspace_destroy(ws);
    return COCONS_ERR_ALLOC;
  }
  if (with_i8 && g_syrk_i8.update && n_pad >= kSyrkI8MinPad &&
      (cudaMalloc(&ws->i8_slices, (size_t)kSyrkI8BytesPerRow * n_pad) != cudaSuccess ||
       cudaMalloc(&ws->i8_scale, sizeof(double) * n_pad) != cudaSuccess)) {
    chol_workspace_destroy(ws);
    return COCONS_ERR_ALLOC;
  }
  return 0;
}

void chol_workspace_destroy(CholWorkspace* ws) {
  cudaFree(ws->winv), cudaFree(ws->info);
  if (ws->i8_slices) cudaFree(ws->i8_slices);
  if (ws->i8_scale) cudaFree(ws->i8_scale);
  ws->i8_slices = nullptr, ws->i8_scale = nullptr;
  if (ws->panel_stream) cudaStreamDestroy(ws->panel_stream);
  if (ws->ev_a) cudaEventDestroy(ws->ev_a);
  if (ws->ev_p) cudaEventDestroy(ws->ev_p);
  if (ws->ev_k0) cudaEventDestroy(ws->ev_k0);
  if (ws->ev_k1) cudaEventDestroy(ws->ev_k1);
  ws->ev_k0 = nullptr, ws->ev_k1 = nullptr;
  ws->winv = nullptr, ws->info = nullptr, ws->panel_stream = nullptr, ws->ev_a = nullptr, ws->ev_p = nullptr;
}

// one outer panel: tiles [J0, J0+jb), every 128-wide step on stream `st`
void factor_panel(double* A, int64_t n_pad, int64_t ld, const CholWorkspace& ws, int64_t J0, int64_t jb,
                  cudaStream_t st) {
  for (int64_t jj = J0; jj < J0 + jb; ++jj) {
    double* Ajj = A + jj * kTile * ld + jj * kTile;
    double* Wjj = ws.winv + jj * (int64_t)kTile * kTile;
    launch_potrf_tile(Ajj, ld, Wjj, ws.info, (int)(jj * kTile), st);
    const int64_t below = n_pad - (jj + 1) * kTile;
    if (below <= 0) continue;
    double* panel = Ajj + kTile;  // rows below the diagonal tile, 128 columns
    // X = A * W^T  (in place: a CTA reads all of its 128 x 128 block before writing it)
    launch_gemm_nt(1, below, kTile, kTile, panel, ld, Wjj, kTile, panel, ld, 0, st);
    const int64_t rest = (J0 + jb - jj - 1) * kTile;  // remaining columns of this outer panel
    if (rest > 0) launch_gemm_nt(0, below, rest, kTile, panel, ld, panel, ld, Ajj + kTile * ld + kTile, ld, 1, st);
  }
}

// Look-ahead: the update by panel J is split into (a) the columns of panel J+1 and (b) everything
// to their right.  As soon as (a) is done, panel J+1 is factored on a high-priority side stream
// while (b) - where the flops are - keeps the SMs busy on the main stream.
// tiles per outer panel: trailing updates run with K = 128 * chol_outer(n_pad).  Measured on B200 at
// n = 50 000: K = 512 -> 1209.7 ms, 768 -> 1200.1, 1024 -> 1199.6 (the read-modify-write epilogue of C is
// amortised over a longer K; standalone SYRK 35.19 / 35.50 / 35.65 TFLOP/s); below ~16 k sites the longer
// panel chain costs more than it saves.  COCONS_CHOL_OUTER overrides.
int chol_outer(int64_t n_pad) {
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("COCONS_CHOL_OUTER");
    forced = e ? std::max(1, std::min(atoi(e), 16)) : 0;
  }
  if (forced > 0) return forced;
  // holes (n_pad = 5632), 8 evaluations in flight: 2 -> 300.9, 3 -> 296.4, 4 -> 288.9 evals/s; stripes (12 032): 4 best
  return n_pad >= 16384 ? 6 : (n_pad >= 8192 ? 4 : 2);
}

// trailing updates with at least this many rows run as split-int8 products (syrk_i8.cu) when the workspace has
// the slices; COCONS_SYRK_I8=0, read on every call, keeps every update on the DMMA GEMM.  Stand-alone lower-triangle
// updates on B200 (tools/syrk_i8_bench.py): int8 / DMMA time 1.24 at 4096 rows, 1.02 at 8192, 0.96 at 16 384
constexpr int64_t kSyrkI8MinRows = 16384;

static bool syrk_i8_enabled(const CholWorkspace& ws) {
  if (!g_syrk_i8.update || !ws.i8_slices) return false;
  const char* e = getenv("COCONS_SYRK_I8");
  return !(e && atoi(e) == 0);
}

int chol_factor(double* A, int64_t n_pad, int64_t ld, CholWorkspace ws, cudaStream_t st) {
  cudaMemsetAsync(ws.info, 0, sizeof(int), st);
  const bool i8 = syrk_i8_enabled(ws);
  const int64_t nt = n_pad / kTile;
  const int64_t outer = chol_outer(n_pad);
  static int lookahead = -1;  // COCONS_CHOL_LOOKAHEAD=0: panel work on the main stream too (debugging knob)
  if (lookahead < 0) {
    const char* e = getenv("COCONS_CHOL_LOOKAHEAD");
    lookahead = e ? atoi(e) : 1;
  }
  cudaStream_t ps = lookahead ? ws.panel_stream : st;
  factor_panel(A, n_pad, ld, ws, 0, std::min<int64_t>(outer, nt), st);
  for (int64_t J0 = 0; J0 < nt; J0 += outer) {
    const int64_t jb = std::min<int64_t>(outer, nt - J0);
    const int64_t done = (J0 + jb) * kTile;
    const int64_t trail = n_pad - done;
    if (trail <= 0) break;
    const int64_t nb_next = std::min<int64_t>(outer, nt - (J0 + jb));
    const int64_t wnext = nb_next * kTile;
    const double* P = A + J0 * kTile * ld + done;  // rows [done, n_pad) of panel J
    const int64_t rest = trail - wnext;
    const bool split = i8 && jb * kTile == kSyrkI8K && trail >= kSyrkI8MinRows;
    if (split) {  // (a) from the slices of all rows of panel J; (b) re-uses them
      g_syrk_i8.split(P, ld, trail, ws.i8_slices, ws.i8_scale, st);
      g_syrk_i8.update(trail, wnext, ws.i8_slices, ws.i8_scale, 0, 0, A + done * ld + done, ld, 1, ws.info, st);
    } else {
      launch_gemm_nt(0, trail, wnext, jb * kTile, P, ld, P, ld, A + done * ld + done, ld, 1, st);  // (a)
    }
    cudaEventRecord(ws.ev_a, st);
    cudaStreamWaitEvent(ps, ws.ev_a, 0);
    factor_panel(A, n_pad, ld, ws, J0 + jb, nb_next, ps);
    cudaEventRecord(ws.ev_p, ps);
    if (rest > 0) {  // (b)
      double* C2 = A + (done + wnext) * ld + done + wnext;
      // the first (b) update is the largest of the factorisation: bracket it with events so that its own
      // duration (measured inside the evaluation) is available for the roofline.  On the int8 path the bracket
      // holds what a stand-alone (b) costs, the split of its rows included: that split is repeated inside it
      // (the same slices again, once per factorisation).
      if (J0 == 0) cudaEventRecord(ws.ev_k0, st);
      if (split) {
        if (J0 == 0) g_syrk_i8.split(P + wnext, ld, rest, ws.i8_slices + wnext * kSyrkI8BytesPerRow,
                                     ws.i8_scale + wnext, st);
        g_syrk_i8.update(rest, rest, ws.i8_slices, ws.i8_scale, wnext, wnext, C2, ld, 1, ws.info, st);
      } else {
        const double* P2 = P + wnext;
        launch_gemm_nt(0, rest, rest, jb * kTile, P2, ld, P2, ld, C2, ld, 1, st);
      }
      if (J0 == 0) cudaEventRecord(ws.ev_k1, st);
    }
    cudaStreamWaitEvent(st, ws.ev_p, 0);
  }
  return 0;
}

}  // namespace cocons
