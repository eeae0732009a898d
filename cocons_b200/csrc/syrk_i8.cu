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
//   for the subtraction (the scalings are exact unless they underflow), in a fixed order - the result is bitwise
//   reproducible, independent of the tiling and equal to tools/ozaki_model.py.
//
// Layout of the slices: for every 128-row tile r of P and every 32-column chunk c (24 of them), a 32 KB block of
// the 8 slices, each 128 rows x 32 B in the UMMA K-major SWIZZLE_32B layout (row i at 32 i, 16-byte half h stored
// at h ^ bit 2 of i).  One stage of the update is one chunk: A = the 32 KB block (one bulk copy), B = the 2 KB
// halves of the 8 slices of its 64 rows.  A tile of C is 128 x 64: its 8 int32 accumulators of 128 x 64 fill the
// 512 columns of tensor memory.
//
// Update kernel: persistent, one CTA per SM, warp-specialised (warp 0 feeds the stages, warp 1 issues the MMAs,
// warps 2-9 run the epilogue).  The epilogue drains the accumulators into registers and hands tensor memory back
// before its read-modify-write of C, so that the products of the next tile run under it; the producer runs ahead
// into the next tile's stages meanwhile.  CTAs can form clusters of kCM x kCN tiles (2 x 2: 256 rows x one 128-wide
// block column) that share their operands: the A block of a tile row is multicast to the CTAs of that row, the B
// halves of a tile column to the CTAs of that column, so each SM pulls half of a stage's 48 KB through L2.
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
constexpr int kEpiWarps = 8;                       // two per tensor-memory lane quarter, each half of the columns
constexpr int kEpiBatch = 16;                      // entries of C per thread read before the first of them is written
#ifdef COCONS_I8_PROBE
constexpr int kProbeWarps = 1;  // the probe build's observer of the stage refills
#else
constexpr int kProbeWarps = 0;
#endif
constexpr int kThreads = 32 * (2 + kEpiWarps + kProbeWarps);  // producer warp, MMA warp, epilogue warps (, observer)
constexpr int kSplitThreads = 128;
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
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// a healthy wait ends within tens of microseconds; one that does not (an arrival or byte count that does not add up,
// which would be a bug) sets *info = COCONS_ERR_CUDA and returns false, and the kernel ends instead of hanging
constexpr uint64_t kWaitLimitNs = 2000000000ull;
__device__ __noinline__ bool mbar_wait(uint32_t bar, uint32_t parity, int* info) {
  if (mbar_try(bar, parity)) return true;
  const uint64_t t0 = globaltimer_ns();
  while (!mbar_try(bar, parity))
    if (globaltimer_ns() - t0 > kWaitLimitNs) {
      atomicCAS(info, 0, COCONS_ERR_CUDA);
      return false;
    }
  return true;
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
// the same bytes at the same offset in every CTA of the cluster named in mask, each signalling its own barrier at bar
__device__ __forceinline__ void bulk_g2s_mc(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], "
      "%4;" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar), "h"(mask)
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

// D = A B^T (acc = 0) or D += A B^T
__device__ __forceinline__ void umma_i8(uint32_t dtmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(dtmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc));
}

// The 36 slice products of a chunk in 12 MMAs.  An MMA costs about the same for N = 64 as for N = 256 (measured on
// B200: 128 x 64 x 32 products ran at a quarter of the int8 rate), so the B slices u0 .. u0 + nblk - 1, which lie
// one after the other in the stage (64 rows each), form one operand of N = 64 nblk, and the MMA of A_t writes it at
// tensor-memory column 64 (t + u0 - 2): block u lands on the accumulator of its weight t + u.  The first two MMAs
// cover the 512 columns exactly once (weights 2-5 and 6-9), so in the first chunk of a tile they overwrite and
// everything after them accumulates: the int32 sums are exact, and their order does not change a bit.
struct SlicePairs {
  int t, u0, nblk;
};
constexpr int kMmas = 12;
__host__ __device__ constexpr SlicePairs slice_pairs(int k) {
  constexpr SlicePairs p[kMmas] = {{1, 1, 4}, {1, 5, 4}, {2, 1, 4}, {3, 1, 4}, {4, 1, 4}, {5, 1, 4},
                                   {6, 1, 3}, {7, 1, 2}, {8, 1, 1}, {2, 5, 3}, {3, 5, 2}, {4, 5, 1}};
  return p[k];
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// arrive on the barrier at bar in every CTA of the cluster named in mask once the MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"(mask)
      : "memory");
}

#define TMEM_LD8(taddr, r)                                                                                      \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"                          \
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) \
               : "r"(taddr))

__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// byte offset of (row i, byte b) inside one 128 x 32 B slice of a chunk block
__host__ __device__ __forceinline__ uint32_t sw32_offset(int i, int b) {
  const uint32_t off = (uint32_t)i * kChunk + (uint32_t)b;
  return off ^ (((off >> 7) & 1u) << 4);
}

}  // namespace

// one thread per row, 128 rows (one tile) per block.  A row with a NaN or infinite entry gets the scale NaN (its
// slices are then immaterial): every entry of C in its row and column becomes NaN, as on the DMMA path, and the
// factorisation's pivot check reports the matrix as not positive definite.
__global__ void __launch_bounds__(kSplitThreads) syrk_i8_split_kernel(const double* __restrict__ P, int64_t ld,
                                                                  int8_t* __restrict__ q, double* __restrict__ scale) {
  const int i = threadIdx.x;
  const int64_t tile = blockIdx.x, row = tile * kRowsA + i;
  const double* p = P + row;
  // max |P_ik| on the bit patterns, sign cleared: for non-negative doubles the integer order is the numeric one, and
  // every NaN lies above infinity - unlike fmax, which skips a NaN
  unsigned long long mb = 0;
  for (int k = 0; k < kSyrkI8K; ++k)
    mb = max(mb, (unsigned long long)__double_as_longlong(p[(int64_t)k * ld]) & 0x7FFFFFFFFFFFFFFFull);
  const double m = __longlong_as_double((long long)mb);
  const bool finite = mb < 0x7FF0000000000000ull;
  int e = 0;
  if (finite && m > 0.0) {
    frexp(m, &e);
    if (ldexp(m, 7 - e) >= 127.5) ++e;
  }
  scale[row] = finite ? ldexp(1.0, e) : __longlong_as_double(0x7FF8000000000000ll);
  // x = P_ik 2^-e as (P_ik f0) f1, both products exact: for a row maximum below 2^-1000, where 2^-e overflows or
  // comes close, 2^-e = 2^64 2^(-e-64); otherwise f0 = 1 and f1 = 2^-e.  (ldexp(P_ik, -e) gives the same bits but
  // compiles to a branchy sequence that kept the loads of the loop below from being unrolled: 5 % slower.)
  const int e0 = e < -1000 ? 64 : 0;
  const double f0 = ldexp(1.0, e0), f1 = ldexp(1.0, -e - e0);
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
          double x = __dmul_rn(__dmul_rn(p[(int64_t)(c * kChunk + 16 * h + 4 * k4 + kb) * ld], f0), f1);
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

namespace {

// Cluster shape in tiles: kCM tile rows (A blocks) x kCN tile columns (B halves).  Measured on B200 (DESIGN.md §3
// K5i): at full clock a tile costs the same ~42 k cycles per SM in every shape - the feed does not bound it - but
// clusters of 4 leave 16 of the 148 SMs unused, and inside a factorisation, which runs at the power limit, sharing
// the B halves (1 x 2) draws less power and keeps a higher clock than 1 x 1.  Other shapes build for comparison.
#ifndef COCONS_I8_CLUSTER_M
#define COCONS_I8_CLUSTER_M 1
#endif
#ifndef COCONS_I8_CLUSTER_N
#define COCONS_I8_CLUSTER_N 2
#endif
constexpr int kCM = COCONS_I8_CLUSTER_M, kCN = COCONS_I8_CLUSTER_N, kCtas = kCM * kCN;
static_assert((kCM == 1 || kCM == 2) && (kCN == 1 || kCN == 2), "clusters of 1 or 2 tile rows and columns");
// super-tiles of 128 kCM rows x 64 kCN columns, numbered by tile_order.cuh: kW of their columns per row unit (with
// lower_only, super-tile (R, C) exists when R >= C / kW, i.e. when it holds at least one lower tile), bands of
// 4096 rows
constexpr int kW = 2 * kCM / kCN, kBand = kBandRows / kCM;

// Probe build (-DCOCONS_I8_PROBE, tools/syrk_i8_probe.py): per-CTA cycle counts summed over the launch
#ifdef COCONS_I8_PROBE
__device__ unsigned long long g_i8_probe[9];  // start->first MMA, MMA full waits, producer empty waits, epilogue,
                                              // MMA waits for tensor memory, CTA cycles, tiles, CTAs, stage refills
#define I8_PROBE(...) __VA_ARGS__
#else
#define I8_PROBE(...)
#endif

__device__ __forceinline__ void super_tile(int64_t st, int ni, int nj, int lower_only, int rm, int cn, int& bi, int& bj,
                                           bool& store) {
  int R, Cc;
  tile_decode<kW, kBand>(st, (ni + kCM - 1) / kCM, nj / kCN, lower_only, R, Cc);
  bi = R * kCM + rm, bj = Cc * kCN + cn;
  // a tile row past the last (odd ni), or a tile above the diagonal blocks of a diagonal super-tile, takes part in
  // feeding its cluster but writes nothing
  store = bi < ni && (!lower_only || bi >= bj / 2);
}

}  // namespace

__global__ void __launch_bounds__(kThreads, 1)
    syrk_i8_update_kernel(int ni, int nj, int lower_only, const int8_t* __restrict__ qa, const double* __restrict__ sa,
                          const int8_t* __restrict__ qb, const double* __restrict__ sb, double* C, int64_t ldc,
                          int* info) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * kStages + 2];
  __shared__ uint32_t tmem_slot;
  I8_PROBE(__shared__ long long issue_t[kStages];)  // clock64 of each stage's copy issue
  I8_PROBE(const long long t_start = clock64();)
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rank = (int)(blockIdx.x % kCtas), rm = rank / kCN, cn = rank % kCN;
  // the clusters (as many as fit the device at once) take the super-tiles in a stride over the banded numbering, so
  // that the tiles in flight stay neighbours
  const int64_t cluster = blockIdx.x / kCtas, nclusters = gridDim.x / kCtas;
  const int64_t nsuper = total_tiles<kW, kBand>((ni + kCM - 1) / kCM, nj / kCN, lower_only);
  const uint32_t stage0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t full0 = smem_u32(bars), empty0 = full0 + 8 * kStages;
  const uint32_t tmem_full = full0 + 16 * kStages, tmem_empty = tmem_full + 8;
  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full0 + 8 * s, 1);         // the local expect_tx; the bytes come from the CTAs that feed this one
      mbar_init(empty0 + 8 * s, kCtas);    // one MMA commit from every CTA of the cluster
    }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 32 * kEpiWarps);
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
  if (kCtas > 1) cluster_sync();  // every barrier of the cluster is initialised before a multicast reaches it
  const uint32_t tmem = tmem_slot;
  I8_PROBE(unsigned long long p_first = 0, p_full = 0, p_empty = 0, p_epi = 0, p_tmem = 0, p_tiles = 0, p_refill = 0;)

  if (warp == 0) {
    if (lane == 0) {
      constexpr uint16_t all = (uint16_t)((1u << kCtas) - 1);
      uint16_t row_mask = 0, col_mask = 0;  // the CTAs that share this CTA's A block / B half
      for (int r = 0; r < kCtas; ++r) {
        if (r / kCN == rm) row_mask |= (uint16_t)(1u << r);
        if (r % kCN == cn) col_mask |= (uint16_t)(1u << r);
      }
      (void)all;
      uint32_t it = 0;
      bool ok = true;
      for (int64_t st = cluster; ok && st < nsuper; st += nclusters) {
        int bi, bj;
        bool store;
        super_tile(st, ni, nj, lower_only, rm, cn, bi, bj, store);
        // the missing tile row of an odd ni fetches the last real block, so that nothing is read past the slices
        const int8_t* a = qa + (int64_t)(bi < ni ? bi : ni - 1) * kChunks * kBlockBytes + cn * (kBlockBytes / kCN);
        const int8_t* b = qb + (int64_t)(bj >> 1) * kChunks * kBlockBytes + (bj & 1) * kSliceBytesB;
        for (int c = 0; c < kChunks; ++c, ++it) {
          const uint32_t slot = it % kStages;
          if (it >= kStages) {
            I8_PROBE(const long long t0 = clock64();)
            if (!mbar_wait(empty0 + 8 * slot, ((it / kStages) - 1) & 1, info)) {
              ok = false;
              break;
            }
            I8_PROBE(p_empty += clock64() - t0;)
          }
          const uint32_t fb = full0 + 8 * slot, da = stage0 + slot * kStageBytes, db = da + kSlices * kSliceBytesA;
          I8_PROBE(*(volatile long long*)&issue_t[slot] = clock64();)
          mbar_expect_tx(fb, kStageBytes);
          const uint32_t aoff = cn * (kBlockBytes / kCN);
          if (kCN > 1)
            bulk_g2s_mc(da + aoff, a + (int64_t)c * kBlockBytes, kBlockBytes / kCN, fb, row_mask);
          else
            bulk_g2s(da + aoff, a + (int64_t)c * kBlockBytes, kBlockBytes / kCN, fb);
#pragma unroll
          for (int t = rm; t < kSlices; t += kCM) {
            if (kCM > 1)
              bulk_g2s_mc(db + t * kSliceBytesB, b + (int64_t)c * kBlockBytes + t * kSliceBytesA, kSliceBytesB, fb,
                          col_mask);
            else
              bulk_g2s(db + t * kSliceBytesB, b + (int64_t)c * kBlockBytes + t * kSliceBytesA, kSliceBytesB, fb);
          }
        }
      }
      // the last commits of the cluster's MMAs arrive on this CTA's empty barriers: wait for them before it exits
      for (uint32_t e = 0; ok && e < kStages; ++e, ++it)
        if (it >= kStages) ok = mbar_wait(empty0 + 8 * (it % kStages), ((it / kStages) - 1) & 1, info);
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint16_t all = (uint16_t)((1u << kCtas) - 1);
      uint32_t it = 0, tl = 0;
      bool ok = true;
      for (int64_t st = cluster; ok && st < nsuper; st += nclusters, ++tl) {
        if (tl > 0) {  // the epilogue has drained the previous tile
          I8_PROBE(const long long t0 = clock64();)
          if (!mbar_wait(tmem_empty, (tl - 1) & 1, info)) break;
          I8_PROBE(p_tmem += clock64() - t0;)
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        for (int c = 0; c < kChunks; ++c, ++it) {
          const uint32_t slot = it % kStages;
          I8_PROBE(const long long t0 = clock64();)
          if (!mbar_wait(full0 + 8 * slot, (it / kStages) & 1, info)) {
            ok = false;
            break;
          }
          I8_PROBE(const long long t1 = clock64(); p_full += t1 - t0; if (it == 0) p_first = t1 - t_start;)
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t da = stage0 + slot * kStageBytes, db = da + kSlices * kSliceBytesA;
#pragma unroll
          for (int k = 0; k < kMmas; ++k) {
            const SlicePairs q = slice_pairs(k);
            umma_i8(tmem + (uint32_t)(q.t + q.u0 - 2) * kRowsB, sw32_desc(da + (q.t - 1) * kSliceBytesA),
                    sw32_desc(db + (q.u0 - 1) * kSliceBytesB), idesc_i8(q.nblk), (c > 0 || k >= 2) ? 1u : 0u);
          }
          // the stage is free in every CTA that fed this one once these MMAs have read it
          if (kCtas > 1)
            umma_commit_mc(empty0 + 8 * slot, all);
          else
            umma_commit(empty0 + 8 * slot);
        }
        if (ok) umma_commit(tmem_full);
        I8_PROBE(++p_tiles;)
      }
    }
#ifdef COCONS_I8_PROBE
  } else if (warp == 2 + kEpiWarps) {
    // observer: the cycles from each stage's copy issue to its full barrier completing, whether or not the MMA thread
    // is waiting for it then.  issue_t[slot] is rewritten only after the MMAs have read the stage, long after this
    if (lane == 0) {
      uint32_t it = 0;
      bool ok = true;
      for (int64_t st = cluster; ok && st < nsuper; st += nclusters)
        for (int c = 0; ok && c < kChunks; ++c, ++it) {
          const uint32_t slot = it % kStages;
          ok = mbar_wait(full0 + 8 * slot, (it / kStages) & 1, info);
          if (ok) p_refill += clock64() - *(volatile long long*)&issue_t[slot];
        }
    }
#endif
  } else {
    // epilogue: C_ij -= ((hi 2^-35 + lo 2^-63) s_i) s_j.  Warp w reads tensor-memory lanes (tile rows) 32 (w % 4) ..,
    // columns 32 h .. 32 h + 31 with h = (w - 2) / 4
    const int quarter = warp & 3, h = (warp - 2) >> 2, r = 32 * quarter + lane;
    const uint32_t trow = tmem + ((uint32_t)(32 * quarter) << 16) + (uint32_t)(32 * h);
    uint32_t tl = 0;
    for (int64_t st = cluster; st < nsuper; st += nclusters, ++tl) {
      int bi, bj;
      bool store;
      super_tile(st, ni, nj, lower_only, rm, cn, bi, bj, store);
      double* Cg = C + (int64_t)(bj * kRowsB + 32 * h) * ldc + (int64_t)bi * kRowsA + r;
      if (store)
#pragma unroll 4
        for (int j = 0; j < 32; ++j) asm volatile("prefetch.global.L2 [%0];" ::"l"(Cg + (int64_t)j * ldc));
      if (!mbar_wait(tmem_full, tl & 1, info)) break;
      I8_PROBE(const long long t0 = clock64();)
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      double v[32];
#pragma unroll
      for (int j0 = 0; j0 < 32; j0 += 8) {
        uint32_t acc[kWeights][8];
#pragma unroll
        for (int w = 0; w < kWeights; ++w) TMEM_LD8(trow + (uint32_t)(w * kRowsB + j0), acc[w]);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          int64_t hi = 0, lo = 0;
#pragma unroll
          for (int w = 0; w < kWeights; ++w) {
            const int64_t s = (int64_t)(int32_t)acc[w][jj];
            if (w + 2 <= kHiTop)
              hi = hi * 128 + s;
            else
              lo = lo * 128 + s;
          }
          v[j0 + jj] = (double)hi * 0x1p-35 + (double)lo * 0x1p-63;
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(tmem_empty);  // the next tile's products may overwrite the accumulators now
      if (store) {
        const double si = sa[(int64_t)bi * kRowsA + r];
        const double* sbj = sb + (int64_t)bj * kRowsB + 32 * h;
        // all loads of a batch before its first store: the compiler cannot move a load of C above a store to C (the
        // addresses differ by the runtime ldc), so one load per store would cost one L2 round trip per entry
#pragma unroll
        for (int j0 = 0; j0 < 32; j0 += kEpiBatch) {
          double c[kEpiBatch], s[kEpiBatch];
#pragma unroll
          for (int j = 0; j < kEpiBatch; ++j) c[j] = __ldcs(Cg + (int64_t)(j0 + j) * ldc), s[j] = sbj[j0 + j];
#pragma unroll
          for (int j = 0; j < kEpiBatch; ++j)  // three roundings, never contracted to an FMA: the model's arithmetic
            __stcs(Cg + (int64_t)(j0 + j) * ldc, __dsub_rn(c[j], __dmul_rn(__dmul_rn(v[j0 + j], si), s[j])));
        }
      }
      I8_PROBE(if (tid == 64) p_epi += clock64() - t0;)
    }
  }
  __syncwarp();
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (kCtas > 1) cluster_sync();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols));
  }
  I8_PROBE(if (tid == 32) {
    atomicAdd(&g_i8_probe[0], p_first), atomicAdd(&g_i8_probe[1], p_full), atomicAdd(&g_i8_probe[4], p_tmem);
    atomicAdd(&g_i8_probe[5], (unsigned long long)(clock64() - t_start)), atomicAdd(&g_i8_probe[6], p_tiles);
    atomicAdd(&g_i8_probe[7], 1ull);
  } if (tid == 0) atomicAdd(&g_i8_probe[2], p_empty);
           if (tid == 64) atomicAdd(&g_i8_probe[3], p_epi);
           if (tid == 32 * (2 + kEpiWarps)) atomicAdd(&g_i8_probe[8], p_refill);)
}

namespace {

static_assert(kHiTop == 5 && kSlices == 8, "the epilogue's 2^-35 and 2^-63 are for 8 slices with weights 2..5 high");

void split(const double* P, int64_t ld, int64_t m, int8_t* q, double* scale, cudaStream_t st) {
  if (m <= 0) return;
  note_launch();
  syrk_i8_split_kernel<<<(unsigned)(m / kRowsA), kSplitThreads, 0, st>>>(P, ld, q, scale);
}

void update(int64_t M, int64_t N, const int8_t* q, const double* scale, int64_t a_row0, int64_t b_row0, double* C,
            int64_t ldc, int lower_only, int* info, cudaStream_t st) {
  if (M <= 0 || N <= 0) return;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCtas, attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // persistent: as many clusters as fit the device at once (one CTA per SM), found once per device
  static int max_clusters[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  int clusters = dev < 16 ? max_clusters[dev] : 0;
  if (clusters <= 0) {
    cudaFuncSetAttribute(syrk_i8_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    cfg.gridDim = dim3(kCtas);
    if (cudaOccupancyMaxActiveClusters(&clusters, syrk_i8_update_kernel, &cfg) != cudaSuccess || clusters <= 0) {
      int sms = 0;
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      clusters = sms / kCtas > 0 ? sms / kCtas : 1;
    }
    if (dev < 16) max_clusters[dev] = clusters;
  }
  const int ni = (int)(M / kRowsA), nj = (int)(N / kRowsB);
  const int64_t nsuper = total_tiles<kW, kBand>((ni + kCM - 1) / kCM, nj / kCN, lower_only);
  cfg.gridDim = dim3((unsigned)(kCtas * (nsuper < clusters ? nsuper : clusters)));
  const int8_t* qa = q + a_row0 / kRowsA * kChunks * (int64_t)kBlockBytes;
  const int8_t* qb = q + b_row0 / kRowsA * kChunks * (int64_t)kBlockBytes;
  note_launch();
  cudaLaunchKernelEx(&cfg, syrk_i8_update_kernel, ni, nj, lower_only, qa, scale + a_row0, qb, scale + b_row0, C, ldc,
                     info);
}

struct Register {
  Register() { g_syrk_i8 = SyrkI8Ops{split, update}; }
} register_syrk_i8;

}  // namespace
}  // namespace cocons

#ifdef COCONS_I8_PROBE
// the probe sums of the launches since the last call, then zero (probe build only)
extern "C" int cocons_i8_probe_read(unsigned long long* out) {
  if (cudaMemcpyFromSymbol(out, cocons::g_i8_probe, sizeof(cocons::g_i8_probe)) != cudaSuccess) return -1;
  const unsigned long long zero[9] = {};
  return cudaMemcpyToSymbol(cocons::g_i8_probe, zero, sizeof(zero)) == cudaSuccess ? 0 : -1;
}
#endif
