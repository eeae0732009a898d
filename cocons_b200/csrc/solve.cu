// Post-factorisation kernels (K6/K7): log-determinant, blocked forward
// substitution with many right-hand sides, and the small Gram reductions from
// which the ML / profile / REML quadratic forms are taken.  They replace
//   sum(log(diag(cholS)))                          R/neg2loglikelihood.R:153,208,267
//   forwardsolve(cholS, ., transpose=TRUE, ...)    :145-147, :214-217, :273-275
//   crossprod(.)                                   :148, :157, :214, :276, :285
// All of them are HBM-bound: the factor is streamed once per block of
// right-hand sides (4 n^2 bytes).
#include <cooperative_groups.h>

#include <algorithm>
#include <cstring>
#include <vector>

#include "../../include/cocons_b200.h"
#include "common.cuh"

namespace cg = cooperative_groups;

namespace cocons {

// sum_{i<n} log L_ii, one CTA, fixed summation order (deterministic)
__global__ void __launch_bounds__(1024) logdet_kernel(const double* __restrict__ L, int64_t n, int64_t ld,
                                                      double* __restrict__ out) {
  __shared__ double red[1024];
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += 1024) s += log(L[i * ld + i]);
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = 512; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = red[0];
}

void launch_logdet(const double* L, int64_t n, int64_t ld, double* out, cudaStream_t st) {
  note_launch();
  logdet_kernel<<<1, 1024, 0, st>>>(L, n, ld, out);
}

// ---------------------------------------------------------------------------
// Blocked forward substitution  L Y = B  for NR right-hand sides in ONE cooperative launch:
//   for every tile J:   y_J = inv(L_JJ) b_J ;   b_I -= L_IJ y_J  for every tile row I > J ;  grid sync.
// Every CTA recomputes y_J in shared memory (a 128 x 128 product out of L2) instead of waiting for a
// broadcast, then updates the tile rows it owns (I = J+1+blockIdx.x, stride gridDim.x); CTA 0 stores y_J.
// The n/128 dependent steps cost one grid barrier each instead of one kernel launch each.
// ---------------------------------------------------------------------------
template <int NR>
__global__ void __launch_bounds__(256) fwd_solve_coop_kernel(const double* __restrict__ L, int64_t ld,
                                                             const double* __restrict__ Winv, double* B,
                                                             double* __restrict__ Y, int64_t ldb, int64_t nt, int nr) {
  cg::grid_group grid = cg::this_grid();
  __shared__ double bj[NR][kTile];
  __shared__ double yj[NR][kTile];
  __shared__ double part[NR][256];
  const int tid = threadIdx.x;
  const int row = tid & (kTile - 1), h = tid >> 7;
  for (int64_t J = 0; J < nt; ++J) {
    const int64_t j0 = J * kTile;
    const double* W = Winv + J * (int64_t)kTile * kTile;
    for (int idx = tid; idx < NR * kTile; idx += 256) {
      const int c = idx / kTile, k = idx % kTile;
      bj[c][k] = (c < nr) ? __ldcg(B + (int64_t)c * ldb + j0 + k) : 0.0;  // written by other CTAs: bypass L1
    }
    __syncthreads();
    {  // y = W b: thread (row, half) sums half of the k range of its row
      double acc[NR];
#pragma unroll
      for (int c = 0; c < NR; ++c) acc[c] = 0.0;
      // W is stored with explicit zeros above the diagonal: fixed trip count, 16 loads in flight
      const double* Wp = W + (int64_t)h * (kTile / 2) * kTile + row;
#pragma unroll 16
      for (int k = 0; k < kTile / 2; ++k) {
        const double w = __ldg(Wp + (int64_t)k * kTile);
#pragma unroll
        for (int c = 0; c < NR; ++c) acc[c] = fma(w, bj[c][h * (kTile / 2) + k], acc[c]);
      }
#pragma unroll
      for (int c = 0; c < NR; ++c) part[c][tid] = acc[c];
    }
    __syncthreads();
    if (tid < kTile) {
#pragma unroll
      for (int c = 0; c < NR; ++c) {
        const double y = part[c][tid] + part[c][tid + kTile];
        yj[c][tid] = y;
        if (blockIdx.x == 0 && c < nr) Y[(int64_t)c * ldb + j0 + tid] = y;
      }
    }
    __syncthreads();
    for (int64_t I = J + 1 + blockIdx.x; I < nt; I += gridDim.x) {  // b_I -= L_IJ y_J
      const int64_t i0 = I * kTile;
      double acc[NR];
#pragma unroll
      for (int c = 0; c < NR; ++c) acc[c] = 0.0;
      const double* Lp = L + (j0 + (int64_t)h * (kTile / 2)) * ld + i0 + row;
#pragma unroll 16
      for (int k = 0; k < kTile / 2; ++k) {
        const double l = __ldg(Lp + (int64_t)k * ld);
#pragma unroll
        for (int c = 0; c < NR; ++c) acc[c] = fma(l, yj[c][h * (kTile / 2) + k], acc[c]);
      }
#pragma unroll
      for (int c = 0; c < NR; ++c) part[c][tid] = acc[c];
      __syncthreads();
      if (tid < kTile) {
#pragma unroll
        for (int c = 0; c < NR; ++c)
          if (c < nr) {  // this row block was last updated by ANOTHER CTA (previous step): read it from L2
            double* bp = B + (int64_t)c * ldb + i0 + tid;
            *bp = __ldcg(bp) - (part[c][tid] + part[c][tid + kTile]);
          }
      }
      __syncthreads();
    }
    grid.sync();
  }
}

// ---------------------------------------------------------------------------
// The same substitution WITHOUT a cooperative launch: two ordinary kernels per tile step (y_J = W_J b_J by one
// CTA; b_I -= L_IJ y_J by one CTA per remaining tile row), same arithmetic and summation order as the
// cooperative kernel.  Opt-in (COCONS_SOLVE_COOP=0): written at the end of round 1 to test whether the
// cooperative launch is what makes overlapping evaluations irreproducible (DESIGN.md §4); it costs 2 n/128
// launches per solve instead of one and has not been run on a GPU yet.
// ---------------------------------------------------------------------------
template <int NR>
__global__ void __launch_bounds__(256) fwd_tile_solve_kernel(const double* __restrict__ W, double* __restrict__ B,
                                                             double* __restrict__ Y, int64_t ldb, int64_t j0, int nr) {
  __shared__ double bj[NR][kTile];
  __shared__ double part[NR][256];
  const int tid = threadIdx.x;
  const int row = tid & (kTile - 1), h = tid >> 7;
  for (int idx = tid; idx < NR * kTile; idx += 256) {
    const int c = idx / kTile, k = idx % kTile;
    bj[c][k] = (c < nr) ? __ldcg(B + (int64_t)c * ldb + j0 + k) : 0.0;
  }
  __syncthreads();
  double acc[NR];
#pragma unroll
  for (int c = 0; c < NR; ++c) acc[c] = 0.0;
  const double* Wp = W + (int64_t)h * (kTile / 2) * kTile + row;
#pragma unroll 16
  for (int k = 0; k < kTile / 2; ++k) {
    const double w = __ldg(Wp + (int64_t)k * kTile);
#pragma unroll
    for (int c = 0; c < NR; ++c) acc[c] = fma(w, bj[c][h * (kTile / 2) + k], acc[c]);
  }
#pragma unroll
  for (int c = 0; c < NR; ++c) part[c][tid] = acc[c];
  __syncthreads();
  if (tid < kTile) {
#pragma unroll
    for (int c = 0; c < NR; ++c)
      if (c < nr) Y[(int64_t)c * ldb + j0 + tid] = part[c][tid] + part[c][tid + kTile];
  }
}

template <int NR>
__global__ void __launch_bounds__(256) fwd_tile_update_kernel(const double* __restrict__ L, int64_t ld,
                                                              const double* __restrict__ Y, double* __restrict__ B,
                                                              int64_t ldb, int64_t J, int nr) {
  __shared__ double yj[NR][kTile];
  __shared__ double part[NR][256];
  const int tid = threadIdx.x;
  const int row = tid & (kTile - 1), h = tid >> 7;
  const int64_t j0 = J * kTile, i0 = (J + 1 + blockIdx.x) * kTile;
  for (int idx = tid; idx < NR * kTile; idx += 256) {
    const int c = idx / kTile, k = idx % kTile;
    yj[c][k] = (c < nr) ? __ldcg(Y + (int64_t)c * ldb + j0 + k) : 0.0;
  }
  __syncthreads();
  double acc[NR];
#pragma unroll
  for (int c = 0; c < NR; ++c) acc[c] = 0.0;
  const double* Lp = L + (j0 + (int64_t)h * (kTile / 2)) * ld + i0 + row;
#pragma unroll 16
  for (int k = 0; k < kTile / 2; ++k) {
    const double l = __ldg(Lp + (int64_t)k * ld);
#pragma unroll
    for (int c = 0; c < NR; ++c) acc[c] = fma(l, yj[c][h * (kTile / 2) + k], acc[c]);
  }
#pragma unroll
  for (int c = 0; c < NR; ++c) part[c][tid] = acc[c];
  __syncthreads();
  if (tid < kTile) {
#pragma unroll
    for (int c = 0; c < NR; ++c)
      if (c < nr) {
        double* bp = B + (int64_t)c * ldb + i0 + tid;
        *bp = __ldcg(bp) - (part[c][tid] + part[c][tid + kTile]);
      }
  }
}

template <int NR>
static void launch_fwd_steps(const double* L, int64_t ld, const double* winv, double* B, double* Y, int64_t ldb,
                             int64_t nt, int nr, cudaStream_t st) {
  for (int64_t J = 0; J < nt; ++J) {
    note_launch();
    fwd_tile_solve_kernel<NR><<<1, 256, 0, st>>>(winv + J * (int64_t)kTile * kTile, B, Y, ldb, J * kTile, nr);
    if (J + 1 < nt) {
      note_launch();
      fwd_tile_update_kernel<NR><<<(unsigned)(nt - J - 1), 256, 0, st>>>(L, ld, Y, B, ldb, J, nr);
    }
  }
}

static bool solve_uses_cooperative_launch() {
  static int coop = -1;
  if (coop < 0) {
    const char* e = getenv("COCONS_SOLVE_COOP");
    coop = (e && atoi(e) == 0) ? 0 : 1;
  }
  return coop != 0;
}

template <int NR>
static void launch_fwd_coop(const double* L, int64_t ld, const double* winv, double* B, double* Y, int64_t ldb,
                            int64_t nt, int nr, cudaStream_t st) {
  static int max_blocks[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 16 && max_blocks[dev] == 0) {
    int sms = 148, per_sm = 1;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fwd_solve_coop_kernel<NR>, 256, 0);
    max_blocks[dev] = sms * (per_sm > 2 ? 2 : (per_sm < 1 ? 1 : per_sm));
  }
  if (!solve_uses_cooperative_launch()) {
    launch_fwd_steps<NR>(L, ld, winv, B, Y, ldb, nt, nr, st);
    return;
  }
  int grid = (dev < 16) ? max_blocks[dev] : 148;
  if (grid > nt) grid = (int)(nt > 0 ? nt : 1);
  void* args[] = {(void*)&L, (void*)&ld, (void*)&winv, (void*)&B, (void*)&Y, (void*)&ldb, (void*)&nt, (void*)&nr};
  note_launch();
  cudaLaunchCooperativeKernel((void*)fwd_solve_coop_kernel<NR>, dim3(grid), dim3(256), args, 0, st);
}

// L (n_pad x n_pad, lower) Y = B for nrhs columns; on return B holds Y.
// Y scratch is provided by the caller through the upper half of B's allocation:
// B must have room for 2*nrhs columns of ldb doubles.
void forward_solve(const double* L, int64_t n_pad, int64_t ld, const double* winv, double* B, int64_t ldb, int nrhs,
                   cudaStream_t st) {
  const int64_t nt = n_pad / kTile;
  double* Y = B + (int64_t)nrhs * ldb;
  for (int c0 = 0; c0 < nrhs; c0 += 8) {
    const int nr = (nrhs - c0 < 8) ? nrhs - c0 : 8;
    double* Bc = B + (int64_t)c0 * ldb;
    double* Yc = Y + (int64_t)c0 * ldb;
    if (nr == 1)
      launch_fwd_coop<1>(L, ld, winv, Bc, Yc, ldb, nt, nr, st);
    else if (nr == 2)
      launch_fwd_coop<2>(L, ld, winv, Bc, Yc, ldb, nt, nr, st);
    else if (nr <= 4)
      launch_fwd_coop<4>(L, ld, winv, Bc, Yc, ldb, nt, nr, st);
    else
      launch_fwd_coop<8>(L, ld, winv, Bc, Yc, ldb, nt, nr, st);
  }
  cudaMemcpyAsync(B, Y, sizeof(double) * (size_t)nrhs * (size_t)ldb, cudaMemcpyDeviceToDevice, st);
}

// ---------------------------------------------------------------------------
// Dataflow forward substitution (K6b, the default).  The cooperative kernel above pays one grid barrier per
// 128-row step (391 of them at n = 50 000: 7.7 ms against a 1.5 ms HBM floor).  Here the work is cut into
// UNITS - tile row I times a chunk of up to kSolveChunk tile columns [J0, J1), 2 MB of L - handed out through
// a ticket counter to persistent CTAs, and the only synchronisation is the dependency itself:
//   ctrl[1] = front = number of finished tile rows of Y (y_I needs y_{I-1}, so rows finish in order)
//   a unit may consume tile column J once front > J; it accumulates  sum_J L_IJ y_J  for its chunk
//   the unit holding the LAST chunk of row I (J1 == I) adds the partial sums of the row's other chunks in chunk
//   order (a fixed order: results do not depend on the schedule), forms y_I = W_I (b_I - sum), stores it over
//   b_I, and publishes front = I + 1.
// Units are issued in the order of the front value they need (J1), last-chunk units first among equals: every
// unit waits only for units with SMALLER tickets, which are already running or done - no deadlock for any
// number of resident CTAs, so an ordinary launch suffices.  CTAs far behind the front stream L at full
// bandwidth (two batches of 16 loads in flight per thread); the chain front -> L_{I,I-1} y_{I-1} -> W_I t -> front
// is the critical path and is kept short: the row-finishing unit holds its piece of L_{I,I-1} in registers before
// the front arrives, picks y_{I-1} up element by element through an 'unset' bit pattern in Y (one L2 hop instead
// of a flag hop followed by a data hop; Y is a scratch copy of the solution, B receives it too), and has the W_I
// loads (prefetched to L2 when the unit starts) in flight during the reduction.  A dependency wait that does not
// end (a bug) sets ctrl[2] and *info and ends the kernel instead of hanging the device.
// Measured at n = 50 000, one right-hand side: 2.47 ms, 10.15 GB read = 4.1 TB/s (profiles/r02_kernels_ncu.md).
// ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_u32(unsigned* p, unsigned v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
constexpr unsigned kSolveSpinLimit = 1u << 25;  // ~seconds; a healthy wait ends within microseconds
constexpr int kSolveSub = 4;                     // tile columns whose y is staged in shared memory at a time

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const double* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
constexpr unsigned long long kSolveUnset = ~0ull;  // cudaMemset(0xFF): no arithmetic result has this bit pattern

template <int NR>
__global__ void __launch_bounds__(256, (NR == 1) ? 2 : 1)
    fwd_solve_flow_kernel(const double* __restrict__ L, int64_t ld, const double* __restrict__ Winv, double* B, double* Y,
                          int64_t ldb, int nr, unsigned* ctrl, const int* __restrict__ units, unsigned nunits,
                          double* part, int nchunks, int* info) {
  extern __shared__ __align__(16) double fsm[];
  double(*ysm)[kSolveSub * kTile] = reinterpret_cast<double(*)[kSolveSub * kTile]>(fsm);  // staged y / t
  double(*red)[256] = reinterpret_cast<double(*)[256]>(fsm + NR * kSolveSub * kTile);      // (row, half) partials
  double(*rq)[4][kTile] = reinterpret_cast<double(*)[4][kTile]>(fsm + NR * (kSolveSub * kTile + 256));  // quarters
  __shared__ unsigned s_u, s_val;
  __shared__ int s_bad;
  const int tid = threadIdx.x, row = tid & (kTile - 1), h = tid >> 7;
  const int rp = tid & 63, kq = tid >> 6;  // critical-path products: rows 2 rp, 2 rp + 1, columns [32 kq, 32 kq + 32)
  unsigned front_seen = 0;                 // uniform over the CTA

  auto give_up = [&]() {
    atomicExch(ctrl + 2, 1u);
    atomicCAS(info, 0, COCONS_ERR_CUDA);
  };
  // thread 0 polls *word until it is >= need; everybody gets the value seen.  false = gave up (error raised)
  auto wait_for = [&](const unsigned* word, unsigned need, unsigned& seen) -> bool {
    if (tid == 0) {
      unsigned v = ld_acquire_u32(word), spins = 0;
      int bad = 0;
      while (v < need) {
        if (++spins > 64) __nanosleep(32);
        if ((spins & 1023u) == 0 && (spins > kSolveSpinLimit || ld_acquire_u32(ctrl + 2) != 0)) {
          bad = 1;
          break;
        }
        v = ld_acquire_u32(word);
      }
      if (bad) give_up();
      s_val = v, s_bad = bad;
    }
    __syncthreads();
    const bool ok = (s_bad == 0);
    seen = s_val;
    __syncthreads();  // s_val / s_bad may be rewritten by the next wait
    return ok;
  };

  for (;;) {
    if (tid == 0) s_u = atomicAdd(ctrl, 1u);
    __syncthreads();
    const unsigned u = s_u;
    __syncthreads();
    if (u >= nunits) break;
    const int I = units[4 * u], J0 = units[4 * u + 1], J1 = units[4 * u + 2], ch = units[4 * u + 3];
    const bool is_final = (J1 == I);
    const int64_t i0 = (int64_t)I * kTile;
    const double* W = Winv + (int64_t)I * kTile * kTile;
    if (is_final) {  // the two tiles of the critical path towards L2: W_I and L_{I,I-1} (128 KB each, 128 B lines)
      for (int l = tid; l < kTile * 8; l += 256) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(W + (int64_t)l * 16));
        if (I > 0)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(L + ((int64_t)(I - 1) * kTile + (l >> 3)) * ld + i0 + (l & 7) * 16));
      }
    }
    double acc[NR], pre[NR];
#pragma unroll
    for (int c = 0; c < NR; ++c) acc[c] = 0.0, pre[c] = 0.0;
    bool presummed = false;
    // partial sums of the row's earlier chunks, in chunk order (tid < 128 holds row `tid`)
    auto presum = [&]() -> bool {
      unsigned done;
      if (ch > 0 && !wait_for(ctrl + 4 + I, (unsigned)ch, done)) return false;
      if (tid < kTile)
        for (int cc = 0; cc < ch; ++cc) {
          const double* pp = part + ((int64_t)I * nchunks + cc) * kSolveMaxRhs * kTile + tid;
#pragma unroll
          for (int c = 0; c < NR; ++c) pre[c] += __ldcg(pp + c * kTile);
        }
      presummed = true;
      return true;
    };

    // ---- streaming part: tile columns [J0, Js) as the front releases them.  The last tile column of a
    //      row-finishing unit (J = I - 1, the one the front is waiting for) takes the fast path below.
    const int Js = (is_final && I > 0) ? I - 1 : J1;
    int ja = J0;
    while (ja < Js) {
      const int avail = ((int)front_seen < Js) ? (int)front_seen : Js;
      if (avail <= ja) {  // nothing consumable yet: use the wait (row-finishing units), then poll the front
        if (is_final && !presummed && !presum()) return;
        unsigned f;
        if (!wait_for(ctrl + 1, (unsigned)ja + 1, f)) return;
        front_seen = f > front_seen ? f : front_seen;
        continue;
      }
      const int jb = (ja + kSolveSub < avail) ? ja + kSolveSub : avail, nt = jb - ja;
      for (int idx = tid; idx < NR * nt * kTile; idx += 256) {
        const int c = idx / (nt * kTile), k = idx - c * nt * kTile;
        ysm[c][k] = (c < nr) ? __ldcg(Y + (int64_t)c * ldb + (int64_t)ja * kTile + k) : 0.0;
      }
      __syncthreads();
      {  // 4 nt batches of 16 columns per thread, the next batch in flight while the current one is consumed
        const int nb = 4 * nt;
        auto src = [&](int q) { return L + ((int64_t)(ja + (q >> 2)) * kTile + h * (kTile / 2) + (q & 3) * 16) * ld + i0 + row; };
        auto use = [&](const double(&v)[16], int q) {
          const double* yp = &ysm[0][(q >> 2) * kTile + h * (kTile / 2) + (q & 3) * 16];
#pragma unroll
          for (int k = 0; k < 16; ++k)
#pragma unroll
            for (int c = 0; c < NR; ++c) acc[c] = fma(v[k], yp[c * kSolveSub * kTile + k], acc[c]);
        };
        double va[16], vb[16];
        {
          const double* p0 = src(0);
#pragma unroll
          for (int k = 0; k < 16; ++k) va[k] = __ldg(p0 + (int64_t)k * ld);
        }
        for (int q = 0; q < nb; q += 2) {  // nb is even
          const double* p1 = src(q + 1);
#pragma unroll
          for (int k = 0; k < 16; ++k) vb[k] = __ldg(p1 + (int64_t)k * ld);
          use(va, q);
          if (q + 2 < nb) {
            const double* p2 = src(q + 2);
#pragma unroll
            for (int k = 0; k < 16; ++k) va[k] = __ldg(p2 + (int64_t)k * ld);
          }
          use(vb, q + 1);
        }
      }
      __syncthreads();  // ysm is rewritten by the next range
      ja = jb;
    }
#pragma unroll
    for (int c = 0; c < NR; ++c) red[c][tid] = acc[c];
    if (!is_final) {
      __syncthreads();
      if (tid < kTile) {
        double* pp = part + ((int64_t)I * nchunks + ch) * kSolveMaxRhs * kTile + tid;
#pragma unroll
        for (int c = 0; c < NR; ++c) pp[c * kTile] = red[c][tid] + red[c][tid + kTile];
      }
      __syncthreads();
      if (tid == 0) {
        __threadfence();
        atomicAdd(ctrl + 4 + I, 1u);
      }
      continue;
    }
    // ---- row-finishing unit: everything that does not depend on y_{I-1} first
    if (!presummed && !presum()) return;
    double q0[NR], q1[NR];
#pragma unroll
    for (int c = 0; c < NR; ++c) q0[c] = q1[c] = 0.0;
    if (I > 0) {
      double2 lreg[32];  // this thread's piece of L_{I,I-1}, in registers before the front gets here
      const double* Lp = L + ((int64_t)(I - 1) * kTile + 32 * kq) * ld + i0 + 2 * rp;
#pragma unroll
      for (int k = 0; k < 32; ++k) lreg[k] = __ldg(reinterpret_cast<const double2*>(Lp + (int64_t)k * ld));
      // y_{I-1}, element by element as its owner stores it (Y was filled with the 'unset' pattern): one hop
      // instead of a flag round trip followed by a data round trip
      int bad = 0;
      for (int idx = tid; idx < NR * kTile; idx += 256) {
        const int c = idx >> 7, k = idx & (kTile - 1);
        double v = 0.0;
        if (c < nr) {
          const double* yp = Y + (int64_t)c * ldb + (int64_t)(I - 1) * kTile + k;
          unsigned long long bits = ld_relaxed_u64(yp);
          unsigned spins = 0;
          while (bits == kSolveUnset) {
            if ((++spins & 1023u) == 0 && (spins > kSolveSpinLimit || ld_acquire_u32(ctrl + 2) != 0)) {
              bad = 1;
              break;
            }
            bits = ld_relaxed_u64(yp);
          }
          v = __longlong_as_double((long long)bits);
        }
        ysm[c][k] = v;
      }
      if (__syncthreads_or(bad)) {
        if (tid == 0) give_up();
        return;
      }
#pragma unroll
      for (int k = 0; k < 32; ++k)
#pragma unroll
        for (int c = 0; c < NR; ++c) {
          const double y = ysm[c][32 * kq + k];
          q0[c] = fma(lreg[k].x, y, q0[c]);
          q1[c] = fma(lreg[k].y, y, q1[c]);
        }
    }
    asm volatile("" ::: "memory");  // keep the W loads behind the products above (lreg and wreg never live together)
    double2 wreg[32];  // W_I from L2 (prefetched at the start of the unit), in flight during the reduction below
    {
      const double* Wp = W + (int64_t)(32 * kq) * kTile + 2 * rp;
#pragma unroll
      for (int k = 0; k < 32; ++k) wreg[k] = __ldg(reinterpret_cast<const double2*>(Wp + (int64_t)k * kTile));
    }
#pragma unroll
    for (int c = 0; c < NR; ++c) rq[c][kq][2 * rp] = q0[c], rq[c][kq][2 * rp + 1] = q1[c];
    __syncthreads();
    if (tid < kTile) {
#pragma unroll
      for (int c = 0; c < NR; ++c) {
        const double own = red[c][tid] + red[c][tid + kTile];
        const double last = (rq[c][0][tid] + rq[c][1][tid]) + (rq[c][2][tid] + rq[c][3][tid]);
        const double b = (c < nr) ? __ldcg(B + (int64_t)c * ldb + i0 + tid) : 0.0;
        ysm[c][tid] = b - ((pre[c] + own) + last);
      }
    }
    __syncthreads();
    // y_I = W_I t (W has explicit zeros above the diagonal)
#pragma unroll
    for (int c = 0; c < NR; ++c) q0[c] = q1[c] = 0.0;
#pragma unroll
    for (int k = 0; k < 32; ++k)
#pragma unroll
      for (int c = 0; c < NR; ++c) {
        const double t = ysm[c][32 * kq + k];
        q0[c] = fma(wreg[k].x, t, q0[c]);
        q1[c] = fma(wreg[k].y, t, q1[c]);
      }
#pragma unroll
    for (int c = 0; c < NR; ++c) rq[c][kq][2 * rp] = q0[c], rq[c][kq][2 * rp + 1] = q1[c];
    __syncthreads();
    if (tid < kTile) {
#pragma unroll
      for (int c = 0; c < NR; ++c)
        if (c < nr) {
          double y = (rq[c][0][tid] + rq[c][1][tid]) + (rq[c][2][tid] + rq[c][3][tid]);
          // a NaN carried over from b (a NaN payload propagates) may have the 'unset' bits: the row-finishing units
          // would wait for it until kSolveSpinLimit and give up, so publish it as the canonical quiet NaN
          unsigned long long bits;
          memcpy(&bits, &y, sizeof bits);
          if (bits == kSolveUnset) y = __longlong_as_double(0x7FF8000000000000ll);
          Y[(int64_t)c * ldb + i0 + tid] = y;  // what the other units read
          B[(int64_t)c * ldb + i0 + tid] = y;  // the caller's result, in place of b_I
        }
    }
    __syncthreads();
    if (tid == 0) {
      __threadfence();
      st_release_u32(ctrl + 1, (unsigned)I + 1);
    }
    if (front_seen < (unsigned)I + 1) front_seen = (unsigned)I + 1;
  }
}

// The work units of the dataflow substitution for T tile rows, in issue order: 4 ints per unit (tile row I, first
// tile column J0, end J1, chunk index).  Issue order = the front value a unit needs (J1); among equals the
// row-finishing units (J1 == I) first, then by row - so every unit depends only on units issued before it.
// Host-only; also reachable through cocons_debug_solve_units for the CPU test of exactly that property.
int build_solve_units(int64_t T, std::vector<int>* out) {
  struct Unit {
    int I, J0, J1, ch;
  };
  std::vector<Unit> units;
  units.push_back({0, 0, 0, 0});
  for (int I = 1; I < T; ++I)
    for (int ch = 0; ch * kSolveChunk < I; ++ch)
      units.push_back({I, ch * kSolveChunk, std::min((ch + 1) * kSolveChunk, I), ch});
  std::stable_sort(units.begin(), units.end(), [](const Unit& a, const Unit& b) {
    if (a.J1 != b.J1) return a.J1 < b.J1;
    const bool fa = a.J1 == a.I, fb = b.J1 == b.I;
    if (fa != fb) return fa;
    return a.I < b.I;
  });
  out->clear();
  for (const Unit& u : units) out->insert(out->end(), {u.I, u.J0, u.J1, u.ch});
  return (int)units.size();
}

int solve_workspace_create(int64_t n_pad, CholWorkspace* ws) {
  const int T = (int)(n_pad / kTile);
  const int nchunks = (T - 1 + kSolveChunk - 1) / kSolveChunk > 0 ? (T - 1 + kSolveChunk - 1) / kSolveChunk : 1;
  std::vector<int> units;
  build_solve_units(T, &units);
  const size_t nunits = units.size() / 4;
  ws->solve_nunits = (int)nunits, ws->solve_nchunks = nchunks;
  if (cudaMalloc(&ws->solve_ctrl, sizeof(unsigned) * (4 + (size_t)T)) != cudaSuccess ||
      cudaMalloc(&ws->solve_units, sizeof(int) * units.size()) != cudaSuccess ||
      cudaMalloc(&ws->solve_part, sizeof(double) * (size_t)T * nchunks * kSolveMaxRhs * kTile) != cudaSuccess) {
    solve_workspace_destroy(ws);
    return COCONS_ERR_ALLOC;
  }
  if (cudaMemcpy(ws->solve_units, units.data(), sizeof(int) * units.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
    solve_workspace_destroy(ws);
    return COCONS_ERR_CUDA;
  }
  return 0;
}

void solve_workspace_destroy(CholWorkspace* ws) {
  cudaFree(ws->solve_ctrl), cudaFree(ws->solve_units), cudaFree(ws->solve_part);
  ws->solve_ctrl = nullptr, ws->solve_units = nullptr, ws->solve_part = nullptr, ws->solve_nunits = 0;
}

template <int NR>
static void launch_fwd_flow(const double* L, int64_t ld, const CholWorkspace& ws, double* B, double* Y, int64_t ldb,
                            int nr, int64_t T, cudaStream_t st) {
  static int sms[16] = {};
  static bool attr_done[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  constexpr int kSmem = NR * (kSolveSub * kTile + 256 + 4 * kTile) * (int)sizeof(double);
  if (dev < 16 && !attr_done[dev]) {
    cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
    cudaFuncSetAttribute(fwd_solve_flow_kernel<NR>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    attr_done[dev] = true;
  }
  const int nsm = (dev < 16 && sms[dev] > 0) ? sms[dev] : 148;
  const unsigned grid = (unsigned)std::min<int64_t>(ws.solve_nunits, 2 * (int64_t)nsm);
  cudaMemsetAsync(ws.solve_ctrl, 0, sizeof(unsigned) * (4 + (size_t)T), st);
  cudaMemsetAsync(Y, 0xFF, sizeof(double) * (size_t)nr * (size_t)ldb, st);  // every y 'unset' (kSolveUnset)
  note_launch();
  fwd_solve_flow_kernel<NR><<<grid, 256, kSmem, st>>>(L, ld, ws.winv, B, Y, ldb, nr, ws.solve_ctrl, ws.solve_units,
                                                      (unsigned)ws.solve_nunits, ws.solve_part, ws.solve_nchunks,
                                                      ws.info);
}

static bool solve_uses_flow() {
  static int flow = -1;
  if (flow < 0) {
    const char* e = getenv("COCONS_SOLVE_FLOW");  // 0: the cooperative kernel (K6) instead of the dataflow kernel (K6b)
    flow = (e && atoi(e) == 0) ? 0 : 1;
  }
  return flow != 0;
}

void forward_solve_ws(const double* L, int64_t n_pad, int64_t ld, const CholWorkspace& ws, double* B, int64_t ldb,
                      int nrhs, cudaStream_t st) {
  if (!ws.solve_units || !solve_uses_flow()) {
    forward_solve(L, n_pad, ld, ws.winv, B, ldb, nrhs, st);
    return;
  }
  const int64_t T = n_pad / kTile;
  double* Y = B + (int64_t)nrhs * ldb;  // scratch behind the right-hand sides (same contract as forward_solve)
  for (int c0 = 0; c0 < nrhs; c0 += kSolveMaxRhs) {
    const int nr = (nrhs - c0 < kSolveMaxRhs) ? nrhs - c0 : kSolveMaxRhs;
    double* Bc = B + (int64_t)c0 * ldb;
    double* Yc = Y + (int64_t)c0 * ldb;
    if (nr == 1)
      launch_fwd_flow<1>(L, ld, ws, Bc, Yc, ldb, nr, T, st);
    else if (nr == 2)
      launch_fwd_flow<2>(L, ld, ws, Bc, Yc, ldb, nr, T, st);
    else if (nr <= 4)
      launch_fwd_flow<4>(L, ld, ws, Bc, Yc, ldb, nr, T, st);
    else
      launch_fwd_flow<8>(L, ld, ws, Bc, Yc, ldb, nr, T, st);
  }
}

// ---------------------------------------------------------------------------
// G = Y^T Y for a tall n x k block (k <= 16), two deterministic passes.
// ---------------------------------------------------------------------------
constexpr int kGramMaxK = 16;
constexpr int kGramBlocks = 296;

__global__ void __launch_bounds__(256) gram_partial_kernel(const double* __restrict__ Y, int64_t n, int64_t ldy, int k,
                                                           double* __restrict__ partial) {
  __shared__ double red[256];
  const int tid = threadIdx.x;
  for (int a = 0; a < k; ++a)
    for (int b = 0; b <= a; ++b) {
      double s = 0.0;
      for (int64_t i = (int64_t)blockIdx.x * 256 + tid; i < n; i += (int64_t)gridDim.x * 256)
        s = fma(Y[(int64_t)a * ldy + i], Y[(int64_t)b * ldy + i], s);
      red[tid] = s;
      __syncthreads();
      for (int w = 128; w > 0; w >>= 1) {
        if (tid < w) red[tid] += red[tid + w];
        __syncthreads();
      }
      if (tid == 0) partial[(int64_t)blockIdx.x * kGramMaxK * kGramMaxK + a * kGramMaxK + b] = red[0];
      __syncthreads();
    }
}

__global__ void gram_final_kernel(const double* __restrict__ partial, int nblocks, int k, double* __restrict__ G) {
  const int a = threadIdx.x / kGramMaxK, b = threadIdx.x % kGramMaxK;
  if (a >= k || b > a) return;
  double s = 0.0;
  for (int blk = 0; blk < nblocks; ++blk) s += partial[(int64_t)blk * kGramMaxK * kGramMaxK + a * kGramMaxK + b];
  G[a * k + b] = s;
  G[b * k + a] = s;
}

// G (k x k, host layout row-major == column-major by symmetry); scratch: kGramBlocks*256 doubles after G
void launch_gram(const double* Y, int64_t n, int64_t ldy, int k, double* G, cudaStream_t st) {
  double* partial = G + kGramMaxK * kGramMaxK;
  note_launch(2);
  gram_partial_kernel<<<kGramBlocks, 256, 0, st>>>(Y, n, ldy, k, partial);
  gram_final_kernel<<<1, kGramMaxK * kGramMaxK, 0, st>>>(partial, kGramBlocks, k, G);
}

}  // namespace cocons
