// K5i: the K = 768 trailing update of chol_factor, C -= P P^T, as exact products of int8 slices on the tensor
// cores (tcgen05.mma kind::i8), combined in FP64 - an Ozaki-I split product.  Model of the arithmetic, and the
// accuracy measurements that fixed its parameters: tools/ozaki_model.py; DESIGN.md §3 K5.
//
//   Split (syrk_i8_split_kernel): per row i a power of two s_i with max_k |P_ik| 128 / s_i < 127.5, and 8 slices by
//   rounding to nearest, x = P_ik / s_i, y = 128 x, a_t = rint(y), x = y - a_t (exact in FP64; |a_1| <= 127, the
//   other |a_t| <= 64), so that P_ik = s_i (sum_t a_t 2^-7t + r 2^-56), |r| <= 1/2.
//   Product: S_w = sum_{t+u=w} A_t A_u^T for the 8 weights w = 2..9 (36 slice products), each exact in int32
//   (|S_w| < 768 (2 127 64 + 6 64^2) < 2^25), then per entry hi = sum_{w<=5} S_w 2^7(5-w) and lo = sum_{w>5}
//   S_w 2^7(9-w), exact in int64, and C_ij -= ((hi 2^-35 + lo 2^-63) s_i) s_j: one rounding for the sum, one
//   for the subtraction, in a fixed order - the result is bitwise reproducible and independent of the tiling.
//
// Layout of the slices: for every 128-row tile r of P and every 32-column chunk c (24 of them), a 32 KB block of
// the 8 slices, each 128 rows x 32 B in the UMMA K-major SWIZZLE_32B layout (row i at 32 i, 16-byte half h stored
// at h ^ bit 2 of i).  One stage of the update is one chunk: A = the 32 KB block (one bulk copy), B = the 2 KB
// halves of the 8 slices of its 64 rows.  A CTA computes one 128 x 64 tile of C: its 8 int32 accumulators of
// 128 x 64 fill the 512 columns of tensor memory.
#include "../../include/cocons_b200.h"
#include "common.cuh"
#include "tile_order.cuh"

namespace cocons {
namespace {

constexpr int kSlices = 8;
constexpr int kWeights = kSlices;           // w = 2..kSlices+1
constexpr int kHiTop = 5;                   // weights 2..kHiTop form the high int64 word
constexpr int kChunk = 32;                  // K per stage = K of one kind::i8 MMA
constexpr int kChunks = kSyrkI8K / kChunk;  // 24
constexpr int kRowsA = 128, kRowsB = 64;
constexpr uint32_t kSliceBytesA = kRowsA * kChunk;                // 4 KB
constexpr uint32_t kSliceBytesB = kRowsB * kChunk;                // 2 KB
constexpr uint32_t kBlockBytes = kSlices * kSliceBytesA;          // 32 KB per (row tile, chunk)
constexpr uint32_t kStageBytes = kSlices * (kSliceBytesA + kSliceBytesB);  // 48 KB
constexpr int kStages = 4;
constexpr int kThreads = 128;
constexpr int kSmemBytes = kStages * kStageBytes + 1024;  // + alignment of the stages to 1 KB
constexpr int kTmemCols = 512;
static_assert(kWeights * kRowsB <= kTmemCols, "the accumulators must fit tensor memory");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
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

// UMMA shared-memory descriptor, K-major SWIZZLE_32B: 8-row groups 256 B apart (SBO), LBO unused (1), version 1
__device__ __forceinline__ uint64_t sw32_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | (1ull << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46) |
         (6ull << 61);
}
// instruction descriptor, kind::i8: D s32, A and B signed, both K-major, M = 128, N = 64 nblk
__host__ __device__ constexpr uint32_t idesc_i8(int nblk) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(nblk * kRowsB >> 3) << 17) | ((uint32_t)(kRowsA >> 4) << 24);
}

// D (+)= A B^T; the accumulators are cleared beforehand, so every MMA accumulates
__device__ __forceinline__ void umma_i8(uint32_t dtmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, 1, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(dtmem),
      "l"(adesc), "l"(bdesc), "r"(idesc));
}

// The 36 slice products of a chunk in 12 MMAs.  An MMA costs about the same for N = 64 as for N = 256 (measured on
// B200: 128 x 64 x 32 products ran at a quarter of the int8 rate), so the B slices u0 .. u0 + nblk - 1, which lie
// one after the other in the stage (64 rows each), form one operand of N = 64 nblk, and the MMA of A_t writes it at
// tensor-memory column 64 (t + u0 - 2): block u lands on the accumulator of its weight t + u.
struct SlicePairs {
  int t, u0, nblk;
};
constexpr int kMmas = 12;
__host__ __device__ constexpr SlicePairs slice_pairs(int k) {
  constexpr SlicePairs p[kMmas] = {{1, 1, 4}, {2, 1, 4}, {3, 1, 4}, {4, 1, 4}, {5, 1, 4}, {6, 1, 3},
                                   {7, 1, 2}, {8, 1, 1}, {1, 5, 4}, {2, 5, 3}, {3, 5, 2}, {4, 5, 1}};
  return p[k];
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

#define TMEM_LD16(taddr, r)                                                                                      \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, " \
               "[%16];"                                                                                          \
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), \
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]),        \
                 "=r"(r[15])                                                                                     \
               : "r"(taddr))

// byte offset of (row i, byte b) inside one 128 x 32 B slice of a chunk block
__host__ __device__ __forceinline__ uint32_t sw32_offset(int i, int b) {
  const uint32_t off = (uint32_t)i * kChunk + (uint32_t)b;
  return off ^ (((off >> 7) & 1u) << 4);
}

}  // namespace

// one thread per row, 128 rows (one tile) per block
__global__ void __launch_bounds__(kThreads) syrk_i8_split_kernel(const double* __restrict__ P, int64_t ld,
                                                                  int8_t* __restrict__ q, double* __restrict__ scale) {
  const int i = threadIdx.x;
  const int64_t tile = blockIdx.x, row = tile * kRowsA + i;
  const double* p = P + row;
  double m = 0.0;
  for (int k = 0; k < kSyrkI8K; ++k) m = fmax(m, fabs(p[(int64_t)k * ld]));
  int e = 0;
  if (m > 0.0) {
    frexp(m, &e);
    if (ldexp(m, 7 - e) >= 127.5) ++e;
  }
  scale[row] = ldexp(1.0, e);
  const double inv = ldexp(1.0, -e);
  int8_t* qt = q + tile * kChunks * (int64_t)kBlockBytes;
  for (int c = 0; c < kChunks; ++c) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint32_t w[kSlices][4];
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
#pragma unroll
        for (int t = 0; t < kSlices; ++t) w[t][k4] = 0;
#pragma unroll
        for (int kb = 0; kb < 4; ++kb) {
          double x = p[(int64_t)(c * kChunk + 16 * h + 4 * k4 + kb) * ld] * inv;
#pragma unroll
          for (int t = 0; t < kSlices; ++t) {
            const double y = x * 128.0;
            const double a = rint(y);
            x = y - a;
            w[t][k4] |= ((uint32_t)(int)a & 0xFFu) << (8 * kb);
          }
        }
      }
#pragma unroll
      for (int t = 0; t < kSlices; ++t)
        *reinterpret_cast<uint4*>(qt + (int64_t)c * kBlockBytes + t * kSliceBytesA + sw32_offset(i, 16 * h)) =
            make_uint4(w[t][0], w[t][1], w[t][2], w[t][3]);
    }
  }
}

// one 128 x 64 tile of C per CTA; warp 0 lane 0 feeds the stages, warp 1 lane 0 issues the MMAs, all four warps
// run the epilogue (warp w owns tensor-memory lanes, i.e. tile rows, 32 w .. 32 w + 31)
__global__ void __launch_bounds__(kThreads, 1)
    syrk_i8_update_kernel(int ni, int nj, int lower_only, const int8_t* __restrict__ qa, const double* __restrict__ sa,
                          const int8_t* __restrict__ qb, const double* __restrict__ sb, double* C, int64_t ldc) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * kStages + 1];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  int bi, bj;
  tile_decode<2>(blockIdx.x, ni, nj, lower_only, bi, bj);
  const uint32_t stage0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t full0 = smem_u32(bars), empty0 = full0 + 8 * kStages, done = full0 + 16 * kStages;
  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    mbar_init(done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)),
                 "r"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_slot;
  {  // clear the accumulators: warp w its 32 lanes, 32 columns per store
    const uint32_t z = 0;
    const uint32_t lane_base = tmem + ((uint32_t)(32 * warp) << 16);
#pragma unroll 1
    for (int col = 0; col < kTmemCols; col += 32)
      asm volatile(
          "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,"
          "%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1};" ::"r"(lane_base + (uint32_t)col),
          "r"(z)
          : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  }

  if (warp == 0 && lane == 0) {
    const int8_t* a = qa + (int64_t)bi * kChunks * kBlockBytes;
    const int8_t* b = qb + (int64_t)(bj >> 1) * kChunks * kBlockBytes + (bj & 1) * kSliceBytesB;
    for (int c = 0; c < kChunks; ++c) {
      const int slot = c % kStages;
      if (c >= kStages) mbar_wait(empty0 + 8 * slot, (uint32_t)((c / kStages - 1) & 1));
      const uint32_t fb = full0 + 8 * slot, da = stage0 + slot * kStageBytes, db = da + kSlices * kSliceBytesA;
      mbar_expect_tx(fb, kStageBytes);
      bulk_g2s(da, a + (int64_t)c * kBlockBytes, kBlockBytes, fb);
#pragma unroll
      for (int t = 0; t < kSlices; ++t)
        bulk_g2s(db + t * kSliceBytesB, b + (int64_t)c * kBlockBytes + t * kSliceBytesA, kSliceBytesB, fb);
    }
  } else if (warp == 1 && lane == 0) {
    for (int c = 0; c < kChunks; ++c) {
      const int slot = c % kStages;
      mbar_wait(full0 + 8 * slot, (uint32_t)((c / kStages) & 1));
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t da = stage0 + slot * kStageBytes, db = da + kSlices * kSliceBytesA;
#pragma unroll
      for (int k = 0; k < kMmas; ++k) {
        const SlicePairs q = slice_pairs(k);
        umma_i8(tmem + (uint32_t)(q.t + q.u0 - 2) * kRowsB, sw32_desc(da + (q.t - 1) * kSliceBytesA),
                sw32_desc(db + (q.u0 - 1) * kSliceBytesB), idesc_i8(q.nblk));
      }
      umma_commit(empty0 + 8 * slot);  // the stage is free once these MMAs have read it
    }
    umma_commit(done);
  }
  __syncwarp();

  // epilogue: C_ij -= ((hi 2^-35 + lo 2^-63) s_i) s_j, 16 columns at a time
  mbar_wait(done, 0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const int r = 32 * warp + lane;
  const double si = sa[(int64_t)bi * kRowsA + r];
  double* Cg = C + (int64_t)bj * kRowsB * ldc + (int64_t)bi * kRowsA + r;
  const double* sbj = sb + (int64_t)bj * kRowsB;
  const uint32_t trow = tmem + ((uint32_t)(32 * warp) << 16);
#pragma unroll 1
  for (int j0 = 0; j0 < kRowsB; j0 += 16) {
    uint32_t acc[kWeights][16];
#pragma unroll
    for (int w = 0; w < kWeights; ++w) TMEM_LD16(trow + (uint32_t)(w * kRowsB + j0), acc[w]);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int jj = 0; jj < 16; ++jj) {
      int64_t hi = 0, lo = 0;
#pragma unroll
      for (int w = 0; w < kWeights; ++w) {
        const int64_t s = (int64_t)(int32_t)acc[w][jj];
        if (w + 2 <= kHiTop)
          hi = hi * 128 + s;
        else
          lo = lo * 128 + s;
      }
      const double v = (double)hi * 0x1p-35 + (double)lo * 0x1p-63;
      double* p = Cg + (int64_t)(j0 + jj) * ldc;
      __stcs(p, __ldcs(p) - (v * si) * sbj[j0 + jj]);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols));
  }
}

namespace {

static_assert(kHiTop == 5 && kSlices == 8, "the epilogue's 2^-35 and 2^-63 are for 8 slices with weights 2..5 high");

void split(const double* P, int64_t ld, int64_t m, int8_t* q, double* scale, cudaStream_t st) {
  if (m <= 0) return;
  note_launch();
  syrk_i8_split_kernel<<<(unsigned)(m / kRowsA), kThreads, 0, st>>>(P, ld, q, scale);
}

void update(int64_t M, int64_t N, const int8_t* q, const double* scale, int64_t a_row0, int64_t b_row0, double* C,
            int64_t ldc, int lower_only, cudaStream_t st) {
  if (M <= 0 || N <= 0) return;
  static bool attr_done[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 16 && !attr_done[dev]) {
    cudaFuncSetAttribute(syrk_i8_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    attr_done[dev] = true;
  }
  const int ni = (int)(M / kRowsA), nj = (int)(N / kRowsB);
  const int64_t tiles = total_tiles<2>(ni, nj, lower_only);
  const int8_t* qa = q + a_row0 / kRowsA * kChunks * (int64_t)kBlockBytes;
  const int8_t* qb = q + b_row0 / kRowsA * kChunks * (int64_t)kBlockBytes;
  note_launch();
  syrk_i8_update_kernel<<<(unsigned)tiles, kThreads, kSmemBytes, st>>>(ni, nj, lower_only, qa, scale + a_row0, qb,
                                                                       scale + b_row0, C, ldc);
}

struct Register {
  Register() { g_syrk_i8 = SyrkI8Ops{split, update}; }
} register_syrk_i8;

}  // namespace
}  // namespace cocons
