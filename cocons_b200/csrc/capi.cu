// C ABI of cocons_b200 (include/cocons_b200.h): host orchestration only - every
// O(n^2) and O(n^3) step is a kernel launch from assembly.cu / chol.cu /
// solve.cu on the context's stream.  No CPU fallback exists: without a usable
// CUDA device every computing entry point returns COCONS_ERR_NO_DEVICE.
#include <algorithm>
#include <atomic>
#include <iterator>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/cocons_b200.h"
#include "common.cuh"

namespace cocons {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static std::atomic<long long> g_launches{0};
void note_launch(int count) { g_launches += count; }

static inline int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

constexpr int kMaxRhs = 16;  // right-hand sides carried through one solve + Gram pass

// ---- small device helpers ------------------------------------------------

// rhs[:, c] = z[:, c] - X mean   (R/neg2loglikelihood.R:210-213), rows >= n are zero
__global__ void residual_kernel(int64_t n, int64_t ld, int p, int nc, const double* __restrict__ X,
                                const double* __restrict__ Z, const double* __restrict__ mean,
                                double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ld) return;
  double trend = 0.0;
  if (i < n && mean)
    for (int k = 0; k < p; ++k) trend = fma(X[(int64_t)k * ld + i], mean[k], trend);
  for (int c = 0; c < nc; ++c) out[(int64_t)c * ld + i] = (i < n) ? Z[(int64_t)c * ld + i] - trend : 0.0;
}

static void launch_residual(int64_t n, int64_t ld, int p, int nc, const double* X, const double* Z, const double* mean,
                            double* out, cudaStream_t st) {
  note_launch();
  residual_kernel<<<(unsigned)((ld + 255) / 256), 256, 0, st>>>(n, ld, p, nc, X, Z, mean, out);
}

// partial sums over a slice of columns k of T (m_pad x n, ld):
//   sto[s][i] = sum_k T(i,k) y_k ,  expl[s][i] = sum_k T(i,k)^2
__global__ void __launch_bounds__(128) pred_reduce_kernel(const double* __restrict__ T, int64_t ld, int64_t m,
                                                          int64_t n, const double* __restrict__ y, int nslices,
                                                          double* __restrict__ sto, double* __restrict__ expl) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const int s = blockIdx.y;
  const int64_t per = (n + nslices - 1) / nslices;
  const int64_t k0 = s * per, k1 = (k0 + per < n) ? k0 + per : n;
  double a = 0.0, b = 0.0;
  for (int64_t k = k0; k < k1; ++k) {
    const double t = T[k * ld + i];
    a = fma(t, y[k], a);
    b = fma(t, t, b);
  }
  sto[(int64_t)s * m + i] = a;
  expl[(int64_t)s * m + i] = b;
}

// out[:, c] = L eps[:, c] for the lower factor, one CTA per tile row (R/sim.R:172, t(eps) %*% R)
template <int NR>
__global__ void __launch_bounds__(128) trmm_lower_kernel(const double* __restrict__ L, int64_t ld,
                                                         const double* __restrict__ E, double* __restrict__ O,
                                                         int64_t lde, int nr) {
  __shared__ double e[NR][kTile];
  const int tid = threadIdx.x;
  const int64_t I = blockIdx.x, i = I * kTile + tid;
  double acc[NR];
#pragma unroll
  for (int c = 0; c < NR; ++c) acc[c] = 0.0;
  for (int64_t J = 0; J <= I; ++J) {
    __syncthreads();
    for (int idx = tid; idx < NR * kTile; idx += 128) {
      const int c = idx / kTile, k = idx % kTile;
      e[c][k] = (c < nr) ? E[(int64_t)c * lde + J * kTile + k] : 0.0;
    }
    __syncthreads();
    const int kend = (J == I) ? tid + 1 : kTile;
    const double* Lp = L + J * kTile * ld + i;
    for (int k = 0; k < kend; ++k) {
      const double l = Lp[(int64_t)k * ld];
#pragma unroll
      for (int c = 0; c < NR; ++c) acc[c] = fma(l, e[c][k], acc[c]);
    }
  }
#pragma unroll
  for (int c = 0; c < NR; ++c)
    if (c < nr) O[(int64_t)c * lde + i] = acc[c];
}

static void launch_trmm_lower(const double* L, int64_t n_pad, int64_t ld, const double* E, double* O, int64_t lde,
                              int k, cudaStream_t st) {
  for (int c0 = 0; c0 < k; c0 += 4) {
    const int nr = (k - c0 < 4) ? k - c0 : 4;
    note_launch();
    trmm_lower_kernel<4><<<(unsigned)(n_pad / kTile), 128, 0, st>>>(L, ld, E + (int64_t)c0 * lde,
                                                                    O + (int64_t)c0 * lde, lde, nr);
  }
}

// ---- host-side small dense algebra (q x q, q <= 16) ----------------------

// in-place lower Cholesky of a k x k row-major matrix; false when not PD
static bool small_chol(std::vector<double>& a, int k) {
  for (int j = 0; j < k; ++j) {
    double d = a[j * k + j];
    for (int t = 0; t < j; ++t) d -= a[j * k + t] * a[j * k + t];
    if (!(d > 0.0)) return false;
    d = std::sqrt(d);
    a[j * k + j] = d;
    for (int i = j + 1; i < k; ++i) {
      double s = a[i * k + j];
      for (int t = 0; t < j; ++t) s -= a[i * k + t] * a[j * k + t];
      a[i * k + j] = s / d;
    }
  }
  return true;
}

// qr(X)$rank as R computes it (LINPACK dqrdc2: Householder with limited column
// pivoting, a column is deferred when its residual norm drops below tol x its
// original norm, tol = 1e-7) - used at R/neg2loglikelihood.R:270.
static int qr_rank_dqrdc2(const double* X, int64_t n, int p, double tol = 1e-7) {
  std::vector<double> a((size_t)n * p);
  std::memcpy(a.data(), X, sizeof(double) * (size_t)n * p);
  std::vector<int> col(p);
  std::vector<double> orig(p);
  auto cnorm = [&](int c, int64_t from) {
    double s = 0;
    for (int64_t i = from; i < n; ++i) s += a[(size_t)c * n + i] * a[(size_t)c * n + i];
    return std::sqrt(s);
  };
  for (int c = 0; c < p; ++c) {
    col[c] = c;
    orig[c] = cnorm(c, 0);
    if (orig[c] == 0) orig[c] = 1;
  }
  int rank = p, k = 0;
  while (k < rank) {
    while (k < rank && cnorm(col[k], k) < tol * orig[col[k]]) {
      const int moved = col[k];
      for (int c = k; c + 1 < p; ++c) col[c] = col[c + 1];
      col[p - 1] = moved;
      --rank;
    }
    if (k >= rank) break;
    const int ck = col[k];
    std::vector<double> v((size_t)(n - k));
    for (int64_t i = k; i < n; ++i) v[(size_t)(i - k)] = a[(size_t)ck * n + i];
    double nrm = 0;
    for (double t : v) nrm += t * t;
    nrm = std::sqrt(nrm);
    if (nrm != 0) {
      v[0] += (v[0] >= 0 ? nrm : -nrm);
      double vn = 0;
      for (double t : v) vn += t * t;
      vn = std::sqrt(vn);
      for (double& t : v) t /= vn;
      for (int c = k; c < p; ++c) {
        const int cc = col[c];
        double dot = 0;
        for (int64_t i = k; i < n; ++i) dot += v[(size_t)(i - k)] * a[(size_t)cc * n + i];
        for (int64_t i = k; i < n; ++i) a[(size_t)cc * n + i] -= 2 * dot * v[(size_t)(i - k)];
      }
    }
    ++k;
  }
  return rank;
}

}  // namespace cocons

using namespace cocons;

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
// debugging aid (COCONS_DEBUG_CHECKSUM=1): deterministic sum of the lower triangle of the n x n matrix
__global__ void __launch_bounds__(256) checksum_partial_kernel(const double* __restrict__ A, int64_t n, int64_t ld,
                                                               double* __restrict__ partial) {
  __shared__ double red[256];
  double s = 0.0;
  for (int64_t j = blockIdx.x; j < n; j += gridDim.x)
    for (int64_t i = j + threadIdx.x; i < n; i += 256) s += A[j * ld + i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = red[0];
}
__global__ void checksum_final_kernel(const double* __restrict__ partial, int nblocks, double* __restrict__ out) {
  double s = 0.0;
  for (int b = 0; b < nblocks; ++b) s += partial[b];
  *out = s;
}

struct cocons_ctx {
  int device = 0;
  int64_t n = 0, n_pad = 0, p = 0, r = 0, q = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::vector<int64_t> perm;  // perm[s] = caller index of sorted site s
  std::vector<double> hX;     // caller-order design (rank computation)
  int rank_x = -1;
  // device
  double *dX = nullptr, *dLocs = nullptr, *dZ = nullptr, *dXb = nullptr;
  double *dTheta = nullptr;  // 6p theta + p mean
  double* dSite = nullptr;
  int* dOrig = nullptr;
  double* dA = nullptr;
  CholWorkspace ws{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  double* dRhs = nullptr;   // n_pad x 2*kMaxRhs
  double* dGram = nullptr;  // Gram + partials + scalars
  // pinned staging
  double* hStage = nullptr;  // theta/mean up, Gram/logdet down
  int* hInfo = nullptr;
  // state of the kept factor
  bool factor_valid = false;
  int mode = 0;
  double nu_fixed = 0, global_range = 1, lim[2] = {0, 0};
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  double ms[4] = {0, 0, 0, 0};
  double kernel_ms = 0, kernel_flops = 0;  // largest trailing-update launch of the last factorisation
  // sparse (tapered) model: spam's CSR pattern (1-based, caller order), the taper values on it, and the
  // caller-index -> sorted-position map
  int *dTapCol = nullptr, *dTapRow = nullptr, *dInv = nullptr;
  double* dTap = nullptr;
  int64_t tap_nnz = 0;
  bool factor_is_taper = false;
  // tiled tapered context (cocons_ctx_create_taper_tiled): only the tiles of L that can be nonzero are stored.
  // Column panel J stacks its tiles column-major: the diagonal tile, the tiles below it (pattern + fill, Morton
  // order), then one right-hand-side tile holding (z - X mean)^T over the panel's columns, so that the factorisation
  // carries the forward substitution along (see tiled_factor).
  bool tiled = false;
  int64_t T = 0, nstored = 0, nfill = 0, tile_products = 0, rhs_k = 0;
  std::vector<int64_t> colptr, rows, base, ldp;  // column starts into rows; tile rows (diagonal first); panel layout
  int64_t g_off = 0;                              // element offset of the Gram block (right-hand sides) in the pool
  std::vector<int64_t> upd_at;                    // per panel: start of its update map in dMaps
  int64_t scat_at = 0;                            // start of the right-hand-side scatter map in dMaps
  double* dPool = nullptr;                        // the stored tiles
  int64_t pool_elems = 0;
  int64_t *dTiles = nullptr, *dMaps = nullptr;    // assembly tile map (TaperSink::tiles); update / scatter maps
  double *dNegI = nullptr, *dLogPart = nullptr;   // -I (128 x rhs_k); log-determinant of each diagonal tile
  double* dCheck = nullptr;  // COCONS_DEBUG_CHECKSUM: 296 partials + [assembly, factor] sums
  double check[2] = {0, 0};
  SiteTable table() const { return SiteTable{dSite, n_pad, dOrig}; }
  TaperTable taper_table() const { return TaperTable{dSite, n_pad}; }  // shares the per-site buffer
};

static int check_device(int device) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_error("no CUDA device available (%s); cocons_b200 has no CPU fallback", cudaGetErrorString(e));
    return COCONS_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= count) {
    set_error("device %d out of range (0..%d)", device, count - 1);
    return COCONS_ERR_ARG;
  }
  cudaDeviceProp prop;
  COCONS_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    return COCONS_ERR_NO_DEVICE;
  }
  COCONS_CUDA_TRY(cudaSetDevice(device));
  return 0;
}

// Evaluations of different contexts may overlap on one device: every context owns its stream, matrix and
// workspace and nothing is shared between their kernel chains.  (Round 1 serialised them behind a per-device
// lock because overlapping chains gave irreproducible factors; the cause was the slot release of the GEMM
// pipeline, csrc/chol.cu, fixed in round 2 - tests/test_gpu_repro.py pins the behaviour.)

// device of the stateless / one-shot entry points: COCONS_DEVICE (one R worker per GPU sets it), default 0
static int default_device() {
  const char* env = getenv("COCONS_DEVICE");
  return env ? atoi(env) : 0;
}

// upload a caller-order n x k column-major host matrix into a sorted, zero-padded n_pad x k device matrix
static int upload_sorted(cocons_ctx* c, const double* src, int64_t k, double* dst) {
  std::vector<double> tmp((size_t)c->n_pad * k, 0.0);
  for (int64_t col = 0; col < k; ++col)
    for (int64_t s = 0; s < c->n; ++s) tmp[(size_t)col * c->n_pad + s] = src[(size_t)col * c->n + c->perm[s]];
  COCONS_CUDA_TRY(cudaMemcpyAsync(dst, tmp.data(), sizeof(double) * tmp.size(), cudaMemcpyHostToDevice, c->stream));
  COCONS_CUDA_TRY(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" {

int cocons_version(void) { return 100; }
long long cocons_launch_count(void) { return g_launches.load(); }
const char* cocons_last_error(void) { return g_err; }
int cocons_device_count(void) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) return 0;
  return count;
}

int cocons_qr_rank(const double* X, int64_t n, int64_t p, double tol) {
  if (!X || n <= 0 || p <= 0 || p > 4096) {
    set_error("qr_rank: bad argument");
    return COCONS_ERR_ARG;
  }
  return qr_rank_dqrdc2(X, n, (int)p, tol);
}

double cocons_sumsmoothlone(const double* x, int64_t len, double lambda, double alpha) {
  // src/cocons_full.cpp:12-30
  double sum = 0;
  for (int64_t w = 0; w < len; ++w) {
    if (std::abs(x[w]) > 1e-4)
      sum = sum + std::abs(x[w]);
    else
      sum = sum + std::pow(alpha, -1) * (std::log(1 + std::exp(-alpha * x[w])) + std::log(1 + std::exp(alpha * x[w])));
  }
  return lambda * sum;
}

// ---- stateless covariance builders ----------------------------------------

static int cov_square(int par, int64_t n, int64_t p, const double* locs, const double* X, const double* theta6,
                      const double* limits, double* out) {
  if (n <= 0 || p <= 0 || !locs || !X || !theta6 || !out) {
    set_error("cov_rns: bad argument");
    return COCONS_ERR_ARG;
  }
  int rc = check_device(default_device());
  if (rc) return rc;
  const double lim[2] = {limits ? limits[0] : 0.0, limits ? limits[1] : 0.0};
  double nu_fixed;
  const int mode = smooth_mode_for(par, (int)p, theta6, lim, &nu_fixed);
  const double global_range = 1 / std::exp(-2 * theta6[p]);  // :62
  cudaStream_t st = nullptr;
  double *dX = nullptr, *dL = nullptr, *dT = nullptr, *dS = nullptr, *dC = nullptr;
  auto cleanup = [&]() {
    cudaFree(dX), cudaFree(dL), cudaFree(dT), cudaFree(dS), cudaFree(dC);
  };
#define TRY_OR_CLEAN(expr)                                                                       \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      set_error("%s failed: %s", #expr, cudaGetErrorString(_e));                                 \
      cleanup();                                                                                 \
      return (_e == cudaErrorMemoryAllocation) ? COCONS_ERR_ALLOC : COCONS_ERR_CUDA;             \
    }                                                                                            \
  } while (0)
  TRY_OR_CLEAN(cudaMalloc(&dX, sizeof(double) * n * p));
  TRY_OR_CLEAN(cudaMalloc(&dL, sizeof(double) * n * 2));
  TRY_OR_CLEAN(cudaMalloc(&dT, sizeof(double) * 6 * p));
  TRY_OR_CLEAN(cudaMalloc(&dS, sizeof(double) * SF_COUNT * n));
  TRY_OR_CLEAN(cudaMalloc(&dC, sizeof(double) * n * n));
  TRY_OR_CLEAN(cudaMemcpyAsync(dX, X, sizeof(double) * n * p, cudaMemcpyHostToDevice, st));
  TRY_OR_CLEAN(cudaMemcpyAsync(dL, locs, sizeof(double) * n * 2, cudaMemcpyHostToDevice, st));
  TRY_OR_CLEAN(cudaMemcpyAsync(dT, theta6, sizeof(double) * 6 * p, cudaMemcpyHostToDevice, st));
  SiteTable T{dS, n, nullptr};
  launch_site_stage(n, n, (int)p, dX, n, dL, n, dT, lim[0], lim[1], mode, T, st);
  launch_assemble_lower(n, n, T, global_range, nu_fixed, mode, dC, n, st);
  launch_symmetrize(n, dC, n, st);
  TRY_OR_CLEAN(cudaGetLastError());
  TRY_OR_CLEAN(cudaMemcpyAsync(out, dC, sizeof(double) * n * n, cudaMemcpyDeviceToHost, st));
  TRY_OR_CLEAN(cudaStreamSynchronize(st));
  cleanup();
  return 0;
}

int cocons_cov_rns(int64_t n, int64_t p, const double* locs, const double* X, const double* theta6,
                   const double* smooth_limits, double* out) {
  if (!smooth_limits) {
    set_error("cov_rns: smooth_limits is required");
    return COCONS_ERR_ARG;
  }
  return cov_square(COCONS_PAR_DIFF, n, p, locs, X, theta6, smooth_limits, out);
}

int cocons_cov_rns_classic(int64_t n, int64_t p, const double* locs, const double* X, const double* theta6,
                           double* out) {
  return cov_square(COCONS_PAR_CLASSIC, n, p, locs, X, theta6, nullptr, out);
}

int cocons_cov_rns_pred(int64_t n, int64_t m, int64_t p, const double* locs, const double* locs_pred, const double* X,
                        const double* X_pred, const double* theta6, const double* limits, double* out) {
  if (n <= 0 || m <= 0 || p <= 0 || !locs || !locs_pred || !X || !X_pred || !theta6 || !limits || !out) {
    set_error("cov_rns_pred: bad argument");
    return COCONS_ERR_ARG;
  }
  int rc = check_device(default_device());
  if (rc) return rc;
  const double global_range = 1 / std::exp(-2 * theta6[p]);  // :351
  cudaStream_t st = nullptr;
  double *dX = nullptr, *dL = nullptr, *dXp = nullptr, *dLp = nullptr, *dT = nullptr, *dS = nullptr, *dSp = nullptr,
         *dC = nullptr;
  auto cleanup = [&]() {
    cudaFree(dX), cudaFree(dL), cudaFree(dXp), cudaFree(dLp), cudaFree(dT), cudaFree(dS), cudaFree(dSp), cudaFree(dC);
  };
  TRY_OR_CLEAN(cudaMalloc(&dX, sizeof(double) * n * p));
  TRY_OR_CLEAN(cudaMalloc(&dL, sizeof(double) * n * 2));
  TRY_OR_CLEAN(cudaMalloc(&dXp, sizeof(double) * m * p));
  TRY_OR_CLEAN(cudaMalloc(&dLp, sizeof(double) * m * 2));
  TRY_OR_CLEAN(cudaMalloc(&dT, sizeof(double) * 6 * p));
  TRY_OR_CLEAN(cudaMalloc(&dS, sizeof(double) * SF_COUNT * n));
  TRY_OR_CLEAN(cudaMalloc(&dSp, sizeof(double) * SF_COUNT * m));
  TRY_OR_CLEAN(cudaMalloc(&dC, sizeof(double) * n * m));
  TRY_OR_CLEAN(cudaMemcpyAsync(dX, X, sizeof(double) * n * p, cudaMemcpyHostToDevice, st));
  TRY_OR_CLEAN(cudaMemcpyAsync(dL, locs, sizeof(double) * n * 2, cudaMemcpyHostToDevice, st));
  TRY_OR_CLEAN(cudaMemcpyAsync(dXp, X_pred, sizeof(double) * m * p, cudaMemcpyHostToDevice, st));
  TRY_OR_CLEAN(cudaMemcpyAsync(dLp, locs_pred, sizeof(double) * m * 2, cudaMemcpyHostToDevice, st));
  TRY_OR_CLEAN(cudaMemcpyAsync(dT, theta6, sizeof(double) * 6 * p, cudaMemcpyHostToDevice, st));
  SiteTable T{dS, n, nullptr}, P{dSp, m, nullptr};
  launch_site_stage(n, n, (int)p, dX, n, dL, n, dT, limits[0], limits[1], SM_GENERAL, T, st);
  launch_site_stage(m, m, (int)p, dXp, m, dLp, m, dT, limits[0], limits[1], SM_GENERAL, P, st);
  launch_assemble_cross(m, n, P, T, global_range, dC, m, st);
  TRY_OR_CLEAN(cudaGetLastError());
  TRY_OR_CLEAN(cudaMemcpyAsync(out, dC, sizeof(double) * n * m, cudaMemcpyDeviceToHost, st));
  TRY_OR_CLEAN(cudaStreamSynchronize(st));
  cleanup();
  return 0;
}

// ---- context ---------------------------------------------------------------

void cocons_ctx_destroy(cocons_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaFree(c->dX), cudaFree(c->dLocs), cudaFree(c->dZ), cudaFree(c->dXb), cudaFree(c->dTheta), cudaFree(c->dSite);
  cudaFree(c->dOrig), cudaFree(c->dA), cudaFree(c->dRhs);
  cudaFree(c->dTapCol), cudaFree(c->dTapRow), cudaFree(c->dInv), cudaFree(c->dTap), cudaFree(c->dCheck);
  cudaFree(c->dPool), cudaFree(c->dTiles), cudaFree(c->dMaps), cudaFree(c->dNegI), cudaFree(c->dLogPart);
  solve_workspace_destroy(&c->ws);
  chol_workspace_destroy(&c->ws);
  cudaFree(c->dGram);
  if (c->hStage) cudaFreeHost(c->hStage);
  if (c->hInfo) cudaFreeHost(c->hInfo);
  for (auto& e : c->ev)
    if (e) cudaEventDestroy(e);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

#define CTX_TRY(expr)                                                                 \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      set_error("%s failed: %s", #expr, cudaGetErrorString(_e));                      \
      cocons_ctx_destroy(c);                                                          \
      return (_e == cudaErrorMemoryAllocation) ? COCONS_ERR_ALLOC : COCONS_ERR_CUDA;  \
    }                                                                                 \
  } while (0)

// tiled: no n_pad^2 matrix and no dense solve workspace (the tiled context allocates its tile pool itself)
static int ctx_create(int device, int64_t n, int64_t p, int64_t r, const double* locs, const double* X,
                      const double* z, void* stream, bool tiled, cocons_ctx** out) {
  int rc = check_device(device);
  if (rc) return rc;
  cocons_ctx* c = new cocons_ctx();
  c->tiled = tiled;
  c->device = device;
  c->n = n, c->p = p, c->r = r;
  c->n_pad = round_up(n, kTile);
  if (stream) {
    c->stream = (cudaStream_t)stream;
  } else {
    CTX_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    c->own_stream = true;
  }
  c->perm.resize((size_t)n);
  morton_order(n, locs, c->perm.data());
  c->hX.assign(X, X + (size_t)n * p);
  const int64_t np = c->n_pad;
  CTX_TRY(cudaMalloc(&c->dX, sizeof(double) * np * p));
  CTX_TRY(cudaMalloc(&c->dLocs, sizeof(double) * np * 2));
  CTX_TRY(cudaMalloc(&c->dZ, sizeof(double) * np * (r > 0 ? r : 1)));
  CTX_TRY(cudaMalloc(&c->dTheta, sizeof(double) * 7 * p));
  CTX_TRY(cudaMalloc(&c->dSite, sizeof(double) * SF_COUNT * np));
  CTX_TRY(cudaMalloc(&c->dOrig, sizeof(int) * np));
  if (!tiled) CTX_TRY(cudaMalloc(&c->dA, sizeof(double) * np * np));
  if (chol_workspace_create(np, &c->ws, !tiled) != 0 || (!tiled && solve_workspace_create(np, &c->ws) != 0)) {
    set_error("ctx_create: out of device memory for the factorisation workspace");
    cocons_ctx_destroy(c);
    return COCONS_ERR_ALLOC;
  }
  CTX_TRY(cudaMalloc(&c->dRhs, sizeof(double) * np * 2 * kMaxRhs));
  CTX_TRY(cudaMalloc(&c->dGram, sizeof(double) * (kMaxRhs * kMaxRhs * 300 + 16)));
  CTX_TRY(cudaMallocHost(&c->hStage, sizeof(double) * (7 * p + kMaxRhs * kMaxRhs + 16)));
  CTX_TRY(cudaMallocHost(&c->hInfo, sizeof(int)));
  for (auto& e : c->ev) CTX_TRY(cudaEventCreate(&e));
  {
    std::vector<int> orig((size_t)np);
    for (int64_t s = 0; s < np; ++s) orig[(size_t)s] = (s < n) ? (int)c->perm[(size_t)s] : (int)s;
    CTX_TRY(cudaMemcpy(c->dOrig, orig.data(), sizeof(int) * np, cudaMemcpyHostToDevice));
  }
  if ((rc = upload_sorted(c, X, p, c->dX)) || (rc = upload_sorted(c, locs, 2, c->dLocs)) ||
      (r > 0 && (rc = upload_sorted(c, z, r, c->dZ)))) {
    cocons_ctx_destroy(c);
    return rc;
  }
  *out = c;
  return 0;
}

int cocons_ctx_create(int device, int64_t n, int64_t p, int64_t r, const double* locs, const double* X,
                      const double* z, void* stream, cocons_ctx** out) {
  if (!out || n <= 0 || p <= 0 || r < 0 || !locs || !X || (r > 0 && !z)) {
    set_error("ctx_create: bad argument");
    return COCONS_ERR_ARG;
  }
  *out = nullptr;
  return ctx_create(device, n, p, r, locs, X, z, stream, false, out);
}

// the entries that need the dense matrix refuse a tiled context
static int refuse_tiled(cocons_ctx* c, const char* who) {
  if (!c || !c->tiled) return 0;
  set_error("%s: not available on a tiled tapered context (cocons_ctx_create_taper_tiled); it supports "
            "cocons_n2ll_taper, cocons_factor_taper, cocons_ctx_get_factor and cocons_ctx_factor_rows", who);
  return COCONS_ERR_STATE;
}

int cocons_ctx_set_z(cocons_ctx* c, const double* z) {
  if (!c || !z || c->r <= 0) {
    set_error("ctx_set_z: bad argument");
    return COCONS_ERR_ARG;
  }
  cudaSetDevice(c->device);
  return upload_sorted(c, z, c->r, c->dZ);
}

int cocons_ctx_set_xbetas(cocons_ctx* c, int64_t q, const double* xb) {
  if (int rc_ = refuse_tiled(c, "ctx_set_xbetas")) return rc_;
  if (!c || q <= 0 || !xb || q >= kMaxRhs) {
    set_error("ctx_set_xbetas: bad argument (q must be in 1..%d)", kMaxRhs - 1);
    return COCONS_ERR_ARG;
  }
  cudaSetDevice(c->device);
  if (c->dXb) cudaFree(c->dXb), c->dXb = nullptr;
  COCONS_CUDA_TRY(cudaMalloc(&c->dXb, sizeof(double) * c->n_pad * q));
  c->q = q;
  return upload_sorted(c, xb, q, c->dXb);
}

// ---- tiled tapered context: layout and factorisation ----------------------------------------------------------

// Tile-level symbolic Cholesky of the Morton-ordered pattern.  The pattern's lower tiles (entries i >= j of the
// caller's pattern, as the assembly keeps them) give each tile column J its rows below the diagonal; eliminating J
// adds its rows to those of its parent (the first of them), which yields every tile L can fill (the elimination tree).
// Then the pool layout: panel J = [diagonal tile, rows below, right-hand-side tile], column-major, ld = 128 x its
// tiles; the Gram block of the right-hand sides (128 x 128) closes the pool.
static void tile_symbolic(cocons_ctx* c, const int32_t* colindices, const int32_t* rowpointers) {
  const int64_t T = c->n_pad / kTile;
  std::vector<int64_t> inv((size_t)c->n);
  for (int64_t s = 0; s < c->n; ++s) inv[(size_t)c->perm[(size_t)s]] = s;
  std::vector<std::vector<int64_t>> st((size_t)T);
  std::vector<int64_t> keys;
  for (int64_t i = 0; i < c->n; ++i) {  // one caller row at a time: its few distinct tile pairs
    keys.clear();
    const int64_t ti = inv[(size_t)i] / kTile;
    for (int64_t e = rowpointers[i] - 1; e < rowpointers[i + 1] - 1; ++e) {
      const int64_t j = colindices[e] - 1;
      if (i < j) continue;
      const int64_t tj = inv[(size_t)j] / kTile;
      if (ti != tj) keys.push_back(std::min(ti, tj) * T + std::max(ti, tj));
    }
    std::sort(keys.begin(), keys.end());
    keys.erase(std::unique(keys.begin(), keys.end()), keys.end());
    for (int64_t k : keys) st[(size_t)(k / T)].push_back(k % T);
  }
  int64_t pattern = 0;
  for (auto& v : st) {
    std::sort(v.begin(), v.end());
    v.erase(std::unique(v.begin(), v.end()), v.end());
    pattern += (int64_t)v.size();
  }
  std::vector<int64_t> merged;
  for (int64_t J = 0; J < T; ++J) {
    const auto& v = st[(size_t)J];
    if (v.empty()) continue;
    auto& par = st[(size_t)v[0]];
    merged.clear();
    std::set_union(par.begin(), par.end(), v.begin() + 1, v.end(), std::back_inserter(merged));
    par.swap(merged);
  }
  c->T = T;
  c->colptr.assign((size_t)T + 1, 0);
  c->rows.clear(), c->base.assign((size_t)T, 0), c->ldp.assign((size_t)T, 0);
  c->tile_products = 0;
  int64_t off = 0;
  for (int64_t J = 0; J < T; ++J) {
    const int64_t m = (int64_t)st[(size_t)J].size();
    c->colptr[(size_t)J] = (int64_t)c->rows.size();
    c->rows.push_back(J);
    c->rows.insert(c->rows.end(), st[(size_t)J].begin(), st[(size_t)J].end());
    c->tile_products += m * (m + 1) / 2;
    c->ldp[(size_t)J] = (m + 2) * kTile;
    c->base[(size_t)J] = off;
    off += c->ldp[(size_t)J] * kTile;
  }
  c->colptr[(size_t)T] = (int64_t)c->rows.size();
  c->nstored = (int64_t)c->rows.size();
  c->nfill = c->nstored - T - pattern;
  c->g_off = off;
  c->pool_elems = off + (int64_t)kTile * kTile;
}

// position of tile row I inside panel J (0: diagonal, m_J + 1: the right-hand-side tile, I == T)
static int64_t tile_pos(const cocons_ctx* c, int64_t I, int64_t J) {
  const int64_t a = c->colptr[(size_t)J], b = c->colptr[(size_t)J + 1];
  if (I == c->T) return b - a;
  const auto it = std::lower_bound(c->rows.begin() + a, c->rows.begin() + b, I);
  return (it != c->rows.begin() + b && *it == I) ? it - (c->rows.begin() + a) : -1;
}

// The maps of gemm_nt_tma_kernel's tile-mapped update (chol.cu): for panel J with rows B = [tiles below J, T] (T
// stands for the right-hand-side tile), pair (a >= b) of B goes to tile (B[a], B[b]) - in panel B[b], or the Gram
// block when both are right-hand sides.  The scatter map puts the 128 x T*128 block of right-hand sides (transposed)
// into the right-hand-side tile of every panel.
static void tile_maps(cocons_ctx* c, std::vector<int64_t>* maps) {
  maps->clear();
  c->upd_at.assign((size_t)c->T, 0);
  for (int64_t J = 0; J < c->T; ++J) {
    std::vector<int64_t> B(c->rows.begin() + c->colptr[(size_t)J] + 1, c->rows.begin() + c->colptr[(size_t)J + 1]);
    B.push_back(c->T);
    const int64_t mb = (int64_t)B.size();
    c->upd_at[(size_t)J] = (int64_t)maps->size();
    for (int64_t a = 0; a < mb; ++a)
      for (int64_t b = 0; b <= a; ++b) {
        if (B[(size_t)b] == c->T) {
          maps->push_back(c->g_off);
          continue;
        }
        const int64_t pos = tile_pos(c, B[(size_t)a], B[(size_t)b]);  // >= 0: the fill of the symbolic step
        maps->push_back(c->base[(size_t)B[(size_t)b]] + pos * kTile);
      }
    for (int64_t b = 0; b < mb; ++b) maps->push_back(B[(size_t)b] == c->T ? kTile : c->ldp[(size_t)B[(size_t)b]]);
  }
  c->scat_at = (int64_t)maps->size();
  for (int64_t J = 0; J < c->T; ++J) maps->push_back(c->base[(size_t)J] + c->ldp[(size_t)J] - kTile);
  for (int64_t J = 0; J < c->T; ++J) maps->push_back(c->ldp[(size_t)J]);
}

// Right-looking factorisation over the column panels, in order, on the context's stream: every target tile receives
// its updates in one fixed order (bitwise reproducible).  Per panel: POTRF + inverse of the diagonal tile (K3b), the
// panel solve X = A W^T over the contiguous rows below it (K4), then ONE tile-mapped launch of C -= P P^T over the
// lower pairs of its row tiles.  The right-hand-side tile rides along as the last row of every panel: its panel
// solve gives y_J^T = (L^-1 (z - X mean))_J^T, its updates are the forward substitution, and the Gram block gathers
// -sum_J y_J^T y_J.  The log-determinant of each diagonal tile goes to dLogPart[J].
static void tiled_factor(cocons_ctx* c, bool rhs, cudaStream_t st) {
  cudaMemsetAsync(c->ws.info, 0, sizeof(int), st);
  const int64_t np = c->n_pad;
  if (rhs) {
    cudaMemsetAsync(c->dRhs, 0, sizeof(double) * np * c->rhs_k, st);
    launch_residual(c->n, np, (int)c->p, (int)c->r, c->dX, c->dZ, c->dTheta + 6 * c->p, c->dRhs, st);
    // 0 - (-I) R^T: the right-hand sides, transposed, into the right-hand-side tile of every panel (exact)
    launch_gemm_nt(2, kTile, np, c->rhs_k, c->dNegI, kTile, c->dRhs, np, c->dPool,
                   (int64_t)(uintptr_t)(c->dMaps + c->scat_at), 0, st);
  }
  for (int64_t J = 0; J < c->T; ++J) {
    double* P = c->dPool + c->base[(size_t)J];
    const int64_t ld = c->ldp[(size_t)J], below = ld - kTile;
    double* W = c->ws.winv + J * (int64_t)kTile * kTile;
    launch_potrf_tile(P, ld, W, c->ws.info, (int)(J * kTile), st);
    launch_logdet(P, std::min<int64_t>(kTile, c->n - J * kTile), ld, c->dLogPart + J, st);
    launch_gemm_nt(1, below, kTile, kTile, P + kTile, ld, W, kTile, P + kTile, ld, 0, st);
    launch_gemm_nt(2, below, below, kTile, P + kTile, ld, P + kTile, ld, c->dPool,
                   (int64_t)(uintptr_t)(c->dMaps + c->upd_at[(size_t)J]), 1, st);
  }
}

// assembly + factorisation of the context's matrix; leaves events 0..2 recorded
static int assemble_and_factor(cocons_ctx* c, int par, const double* theta6, const double* limits,
                               const double* mean_p, bool taper = false) {
  const int64_t p = c->p, np = c->n_pad;
  const double lim[2] = {limits ? limits[0] : 0.0, limits ? limits[1] : 0.0};
  c->mode = smooth_mode_for(par, (int)p, theta6, lim, &c->nu_fixed);
  c->global_range = 1 / std::exp(-2 * theta6[p]);
  c->lim[0] = lim[0], c->lim[1] = lim[1];
  std::memcpy(c->hStage, theta6, sizeof(double) * 6 * p);
  if (mean_p)
    std::memcpy(c->hStage + 6 * p, mean_p, sizeof(double) * p);
  else
    std::memset(c->hStage + 6 * p, 0, sizeof(double) * p);
  COCONS_CUDA_TRY(cudaMemcpyAsync(c->dTheta, c->hStage, sizeof(double) * 7 * p, cudaMemcpyHostToDevice, c->stream));
  COCONS_CUDA_TRY(cudaEventRecord(c->ev[0], c->stream));
  if (c->tiled) {
    // tiled tapered model: zero pool (fill tiles included), unit diagonal in the padding, taper[e] * cov[e] through
    // the tile map
    const int64_t last = c->T - 1;
    launch_taper_site_stage(c->n, (int)p, c->dX, np, c->dLocs, np, c->dTheta, lim[0], lim[1], c->mode, 0,
                            c->taper_table(), c->stream);
    COCONS_CUDA_TRY(cudaMemsetAsync(c->dPool, 0, sizeof(double) * c->pool_elems, c->stream));
    launch_taper_pad_diag(c->n - last * kTile, kTile, c->dPool + c->base[(size_t)last], c->ldp[(size_t)last],
                          c->stream);
    TaperSink S{TS_TILED, nullptr, c->dTap, c->dInv, c->dPool, c->T, c->nstored, c->dTiles};
    launch_taper_entries(0, c->tap_nnz, c->n, c->dTapCol, c->dTapRow, c->taper_table(), c->taper_table(), 1, c->mode,
                         c->nu_fixed, S, c->stream);
  } else if (taper) {
    // tapered model: zero matrix, then taper[e] * cov[e] scattered onto the pattern (R/neg2loglikelihood.R:26-31)
    launch_taper_site_stage(c->n, (int)p, c->dX, np, c->dLocs, np, c->dTheta, lim[0], lim[1], c->mode, 0,
                            c->taper_table(), c->stream);
    COCONS_CUDA_TRY(cudaMemsetAsync(c->dA, 0, sizeof(double) * np * np, c->stream));
    launch_taper_pad_diag(c->n, np, c->dA, np, c->stream);
    launch_taper_entries(0, c->tap_nnz, c->n, c->dTapCol, c->dTapRow, c->taper_table(), c->taper_table(), 1, c->mode,
                         c->nu_fixed, TaperSink{TS_LOWER, nullptr, c->dTap, c->dInv, c->dA, np, 0}, c->stream);
  } else {
    launch_site_stage(c->n, np, (int)p, c->dX, np, c->dLocs, np, c->dTheta, lim[0], lim[1], c->mode, c->table(),
                      c->stream);
    launch_assemble_lower(c->n, np, c->table(), c->global_range, c->nu_fixed, c->mode, c->dA, np, c->stream);
  }
  c->factor_is_taper = taper;
  static int debug_checksum = -1;
  if (debug_checksum < 0) debug_checksum = getenv("COCONS_DEBUG_CHECKSUM") ? 1 : 0;
  if (debug_checksum && !c->tiled) {
    if (!c->dCheck) COCONS_CUDA_TRY(cudaMalloc(&c->dCheck, sizeof(double) * 304));
    checksum_partial_kernel<<<296, 256, 0, c->stream>>>(c->dA, c->n, np, c->dCheck);
    checksum_final_kernel<<<1, 1, 0, c->stream>>>(c->dCheck, 296, c->dCheck + 300);
  }
  COCONS_CUDA_TRY(cudaEventRecord(c->ev[1], c->stream));
  if (c->tiled)
    tiled_factor(c, c->r > 0, c->stream);
  else
    chol_factor(c->dA, np, np, c->ws, c->stream);
  COCONS_CUDA_TRY(cudaEventRecord(c->ev[2], c->stream));
  if (debug_checksum && !c->tiled) {
    checksum_partial_kernel<<<296, 256, 0, c->stream>>>(c->dA, c->n, np, c->dCheck);
    checksum_final_kernel<<<1, 1, 0, c->stream>>>(c->dCheck, 296, c->dCheck + 301);
    COCONS_CUDA_TRY(cudaMemcpyAsync(c->check, c->dCheck + 300, sizeof(double) * 2, cudaMemcpyDeviceToHost, c->stream));
  }
  COCONS_CUDA_TRY(cudaGetLastError());
  c->factor_valid = false;
  return 0;
}

static int finish_timings(cocons_ctx* c) {
  float a = 0, b = 0, d = 0;
  COCONS_CUDA_TRY(cudaEventElapsedTime(&a, c->ev[0], c->ev[1]));
  COCONS_CUDA_TRY(cudaEventElapsedTime(&b, c->ev[1], c->ev[2]));
  COCONS_CUDA_TRY(cudaEventElapsedTime(&d, c->ev[2], c->ev[3]));
  c->ms[0] = a, c->ms[1] = b, c->ms[2] = d, c->ms[3] = a + b + d;
  c->kernel_ms = 0, c->kernel_flops = 0;
  if (c->tiled) return 0;
  const int64_t outer = chol_outer(c->n_pad);
  const int64_t rest = c->n_pad - 2 * outer * kTile;  // rows/cols right of the first two outer panels
  if (rest > 0) {
    float km = 0;
    if (cudaEventElapsedTime(&km, c->ws.ev_k0, c->ws.ev_k1) == cudaSuccess) {
      const double tiles = 2.0 * ((double)(rest / kTile) * (rest / kTile + 1) / 2.0);  // 128 x 64 tiles computed
      c->kernel_ms = km;
      c->kernel_flops = tiles * 2.0 * 128.0 * 64.0 * (double)(outer * kTile);
    }
  }
  return 0;
}

// what ws.info < 0 means after a factorisation or forward substitution: a dependency wait of the dataflow kernel
// (solve.cu) or a barrier wait of the split-int8 update (syrk_i8.cu) ended at its limit instead of hanging the device
static const char* const kSolveGaveUp =
    "a device wait of the forward substitution or the split-int8 update gave up (COCONS_ERR_CUDA)";

// after the substitutions on the kept factor (prediction, betas): report a wait that gave up, and clear it so that
// the factor - still valid - can be used again
static int solve_status(cocons_ctx* c, const char* who) {
  COCONS_CUDA_TRY(cudaMemcpyAsync(c->hInfo, c->ws.info, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  COCONS_CUDA_TRY(cudaStreamSynchronize(c->stream));
  if (*c->hInfo >= 0) return 0;
  const int rc = *c->hInfo;
  COCONS_CUDA_TRY(cudaMemsetAsync(c->ws.info, 0, sizeof(int), c->stream));
  set_error("%s: %s", who, kSolveGaveUp);
  return rc;
}

static int n2ll_impl(cocons_ctx* c, int kind, const double* theta6, const double* limits, const double* mean_p,
                     double* logdet, double* quad, double* logdet_w, int* rank_x, bool taper) {
  if (!c || !theta6 || !limits || !logdet || !quad || kind < COCONS_ML || kind > COCONS_REML || c->r <= 0) {
    set_error("n2ll: bad argument");
    return COCONS_ERR_ARG;
  }
  if (kind == COCONS_PROFILE && (!c->dXb || c->q <= 0)) {
    set_error("n2ll: COCONS_PROFILE needs cocons_ctx_set_xbetas first");
    return COCONS_ERR_STATE;
  }
  if (kind == COCONS_REML && c->p >= kMaxRhs) {
    set_error("n2ll: REML supports at most %d design columns", kMaxRhs - 1);
    return COCONS_ERR_ARG;
  }
  cudaSetDevice(c->device);
  int rc = assemble_and_factor(c, COCONS_PAR_DIFF, theta6, limits, kind == COCONS_ML ? mean_p : nullptr, taper);
  if (rc) return rc;
  const int64_t np = c->n_pad, p = c->p;
  cudaStream_t st = c->stream;
  double* dLogdet = c->dGram + kMaxRhs * kMaxRhs * 300;
  launch_logdet(c->dA, c->n, np, dLogdet, st);
  // mean-design block solved once (PROFILE: x_betas, REML: the full design; :145-147, :273-275)
  const int qx = (kind == COCONS_PROFILE) ? (int)c->q : (kind == COCONS_REML ? (int)p : 0);
  if (qx > 0) {
    const double* src = (kind == COCONS_PROFILE) ? c->dXb : c->dX;
    COCONS_CUDA_TRY(cudaMemcpyAsync(c->dRhs, src, sizeof(double) * np * qx, cudaMemcpyDeviceToDevice, st));
    forward_solve_ws(c->dA, np, np, c->ws, c->dRhs, np, qx, st);
  }
  const int chunk = kMaxRhs - qx;
  double lw = 0.0;
  for (int64_t c0 = 0; c0 < c->r; c0 += chunk) {
    const int nc = (int)((c->r - c0 < chunk) ? c->r - c0 : chunk);
    double* rhs = c->dRhs + (int64_t)qx * np;
    launch_residual(c->n, np, (int)p, nc, c->dX, c->dZ + c0 * np, kind == COCONS_ML ? c->dTheta + 6 * p : nullptr, rhs,
                    st);
    forward_solve_ws(c->dA, np, np, c->ws, rhs, np, nc, st);
    const int k = qx + nc;
    launch_gram(c->dRhs, c->n, np, k, c->dGram, st);
    if (c0 + nc >= c->r) COCONS_CUDA_TRY(cudaEventRecord(c->ev[3], st));
    double* hG = c->hStage + 7 * p;
    COCONS_CUDA_TRY(cudaMemcpyAsync(hG, c->dGram, sizeof(double) * k * k, cudaMemcpyDeviceToHost, st));
    COCONS_CUDA_TRY(cudaMemcpyAsync(hG + kMaxRhs * kMaxRhs, dLogdet, sizeof(double), cudaMemcpyDeviceToHost, st));
    COCONS_CUDA_TRY(cudaMemcpyAsync(c->hInfo, c->ws.info, sizeof(int), cudaMemcpyDeviceToHost, st));
    COCONS_CUDA_TRY(cudaStreamSynchronize(st));
    if (*c->hInfo != 0) {
      cudaEventRecord(c->ev[3], st);
      cudaStreamSynchronize(st);
      finish_timings(c);
      if (*c->hInfo < 0) set_error("n2ll: %s", kSolveGaveUp);
      return *c->hInfo;  // > 0: not positive definite
    }
    *logdet = hG[kMaxRhs * kMaxRhs];
    if (qx == 0) {
      for (int j = 0; j < nc; ++j) quad[c0 + j] = hG[j * k + j];
    } else {
      // z'Pz = |y|^2 - b' W^-1 b with W = Yx'Yx, b = Yx'y  (SURVEY.md §8c: identical to the
      // explicit projector route of :149-150 to 1e-14)
      std::vector<double> W((size_t)qx * qx);
      for (int a = 0; a < qx; ++a)
        for (int b = 0; b < qx; ++b) W[(size_t)a * qx + b] = hG[a * k + b];
      if (!small_chol(W, qx)) {
        set_error("n2ll: X' Sigma^-1 X is not positive definite (rank-deficient mean design)");
        return COCONS_ERR_STATE;
      }
      lw = 0.0;
      for (int a = 0; a < qx; ++a) lw += std::log(W[(size_t)a * qx + a]);
      for (int j = 0; j < nc; ++j) {
        std::vector<double> t(qx);
        double bb = 0.0;
        for (int a = 0; a < qx; ++a) {  // forward solve chol(W) t = b
          double s = hG[a * k + (qx + j)];
          for (int b = 0; b < a; ++b) s -= W[(size_t)a * qx + b] * t[b];
          t[a] = s / W[(size_t)a * qx + a];
          bb += t[a] * t[a];
        }
        quad[c0 + j] = hG[(qx + j) * k + (qx + j)] - bb;
      }
    }
  }
  if (logdet_w) *logdet_w = lw;
  if (rank_x) {
    *rank_x = 0;
    if (kind == COCONS_REML) {
      if (c->rank_x < 0) c->rank_x = qr_rank_dqrdc2(c->hX.data(), c->n, (int)p);
      *rank_x = c->rank_x;
    }
  }
  c->factor_valid = true;
  return finish_timings(c);
}

int cocons_n2ll(cocons_ctx* c, int kind, const double* theta6, const double* limits, const double* mean_p,
                double* logdet, double* quad, double* logdet_w, int* rank_x) {
  if (int rc_ = refuse_tiled(c, "n2ll")) return rc_;
  return n2ll_impl(c, kind, theta6, limits, mean_p, logdet, quad, logdet_w, rank_x, false);
}

// ---- sparse (tapered) model -------------------------------------------------

// spam's 1-based CSR slots: rowpointers[0] == 1, non-decreasing, rowpointers[nrows] - 1 == nnz, columns in 1..ncols
static int check_pattern(const char* who, const int32_t* colindices, const int32_t* rowpointers, int64_t nrows,
                         int64_t ncols, int64_t nnz) {
  if (!colindices || !rowpointers || nnz < 0 || nnz > INT32_MAX || rowpointers[0] != 1 ||
      (int64_t)rowpointers[nrows] - 1 != nnz) {
    set_error("%s: malformed pattern (rowpointers must start at 1 and end at nnz + 1)", who);
    return COCONS_ERR_ARG;
  }
  for (int64_t i = 0; i < nrows; ++i)
    if (rowpointers[i + 1] < rowpointers[i]) {
      set_error("%s: rowpointers decrease at row %lld", who, (long long)i + 1);
      return COCONS_ERR_ARG;
    }
  for (int64_t e = 0; e < nnz; ++e)
    if (colindices[e] < 1 || colindices[e] > ncols) {
      set_error("%s: colindices[%lld] = %d outside 1..%lld", who, (long long)e, colindices[e], (long long)ncols);
      return COCONS_ERR_ARG;
    }
  return 0;
}

static int attach_taper(cocons_ctx* c, const int32_t* colindices, const int32_t* rowpointers,
                        const double* taper_entries, int64_t nnz) {
  cudaSetDevice(c->device);
  cudaFree(c->dTapCol), cudaFree(c->dTapRow), cudaFree(c->dTap);
  c->dTapCol = c->dTapRow = nullptr, c->dTap = nullptr, c->tap_nnz = 0;
  COCONS_CUDA_TRY(cudaMalloc(&c->dTapCol, sizeof(int) * std::max<int64_t>(nnz, 1)));
  COCONS_CUDA_TRY(cudaMalloc(&c->dTapRow, sizeof(int) * (c->n + 1)));
  COCONS_CUDA_TRY(cudaMalloc(&c->dTap, sizeof(double) * std::max<int64_t>(nnz, 1)));
  if (!c->dInv) {
    std::vector<int> inv((size_t)c->n);
    for (int64_t s = 0; s < c->n; ++s) inv[(size_t)c->perm[(size_t)s]] = (int)s;
    COCONS_CUDA_TRY(cudaMalloc(&c->dInv, sizeof(int) * c->n));
    COCONS_CUDA_TRY(cudaMemcpy(c->dInv, inv.data(), sizeof(int) * c->n, cudaMemcpyHostToDevice));
  }
  COCONS_CUDA_TRY(cudaMemcpy(c->dTapCol, colindices, sizeof(int) * nnz, cudaMemcpyHostToDevice));
  COCONS_CUDA_TRY(cudaMemcpy(c->dTapRow, rowpointers, sizeof(int) * (c->n + 1), cudaMemcpyHostToDevice));
  COCONS_CUDA_TRY(cudaMemcpy(c->dTap, taper_entries, sizeof(double) * nnz, cudaMemcpyHostToDevice));
  c->tap_nnz = nnz;
  return 0;
}

int cocons_ctx_set_taper(cocons_ctx* c, const int32_t* colindices, const int32_t* rowpointers,
                         const double* taper_entries, int64_t nnz) {
  if (!c || !taper_entries) {
    set_error("ctx_set_taper: bad argument");
    return COCONS_ERR_ARG;
  }
  int rc = refuse_tiled(c, "ctx_set_taper");
  if (rc || (rc = check_pattern("ctx_set_taper", colindices, rowpointers, c->n, c->n, nnz))) return rc;
  return attach_taper(c, colindices, rowpointers, taper_entries, nnz);
}

int cocons_ctx_create_taper_tiled(int device, int64_t n, int64_t p, int64_t r, const double* locs, const double* X,
                                  const double* z, const int32_t* colindices, const int32_t* rowpointers,
                                  const double* taper_entries, int64_t nnz, void* stream, cocons_ctx** out) {
  if (!out || n <= 0 || p <= 0 || r < 0 || r > kTile || !locs || !X || (r > 0 && !z) || !taper_entries) {
    set_error("ctx_create_taper_tiled: bad argument (r must be in 0..%d)", kTile);
    return COCONS_ERR_ARG;
  }
  *out = nullptr;
  int rc = check_pattern("ctx_create_taper_tiled", colindices, rowpointers, n, n, nnz);
  if (rc) return rc;
  cocons_ctx* c = nullptr;
  if ((rc = ctx_create(device, n, p, r, locs, X, z, stream, true, &c))) return rc;
  if ((rc = attach_taper(c, colindices, rowpointers, taper_entries, nnz))) {
    cocons_ctx_destroy(c);
    return rc;
  }
  tile_symbolic(c, colindices, rowpointers);
  std::vector<int64_t> tiles((size_t)(c->T + 1 + 2 * c->nstored + c->T)), maps;
  for (int64_t J = 0; J < c->T; ++J) {
    tiles[(size_t)(c->T + 1 + 2 * c->nstored + J)] = c->ldp[(size_t)J];
    for (int64_t k = c->colptr[(size_t)J]; k < c->colptr[(size_t)J + 1]; ++k)
      tiles[(size_t)(c->T + 1 + c->nstored + k)] = c->base[(size_t)J] + (k - c->colptr[(size_t)J]) * kTile;
  }
  std::copy(c->colptr.begin(), c->colptr.end(), tiles.begin());
  std::copy(c->rows.begin(), c->rows.end(), tiles.begin() + c->T + 1);
  tile_maps(c, &maps);
  c->rhs_k = std::max<int64_t>(16, round_up(r, 16));
  std::vector<double> negi((size_t)kTile * c->rhs_k, 0.0);
  for (int64_t k = 0; k < c->rhs_k; ++k) negi[(size_t)(k * kTile + k)] = -1.0;
  cudaFree(c->dRhs), c->dRhs = nullptr;
  CTX_TRY(cudaMalloc(&c->dRhs, sizeof(double) * c->n_pad * c->rhs_k));
  CTX_TRY(cudaMalloc(&c->dPool, sizeof(double) * c->pool_elems));
  CTX_TRY(cudaMalloc(&c->dTiles, sizeof(int64_t) * tiles.size()));
  CTX_TRY(cudaMalloc(&c->dMaps, sizeof(int64_t) * maps.size()));
  CTX_TRY(cudaMalloc(&c->dNegI, sizeof(double) * negi.size()));
  CTX_TRY(cudaMalloc(&c->dLogPart, sizeof(double) * c->T));
  CTX_TRY(cudaMemcpy(c->dTiles, tiles.data(), sizeof(int64_t) * tiles.size(), cudaMemcpyHostToDevice));
  CTX_TRY(cudaMemcpy(c->dMaps, maps.data(), sizeof(int64_t) * maps.size(), cudaMemcpyHostToDevice));
  CTX_TRY(cudaMemcpy(c->dNegI, negi.data(), sizeof(double) * negi.size(), cudaMemcpyHostToDevice));
  *out = c;
  return 0;
}

int cocons_ctx_tile_stats(cocons_ctx* c, int64_t* stats4) {
  if (!c || !stats4) {
    set_error("ctx_tile_stats: bad argument");
    return COCONS_ERR_ARG;
  }
  if (!c->tiled) {
    set_error("ctx_tile_stats: the context is dense (tile statistics exist for cocons_ctx_create_taper_tiled)");
    return COCONS_ERR_STATE;
  }
  stats4[0] = c->T, stats4[1] = c->nstored, stats4[2] = c->nfill, stats4[3] = c->tile_products;
  return 0;
}

// GetNeg2loglikelihoodTaper on a tiled context: the factorisation already carried the substitution (tiled_factor);
// what is left is reading the Gram block's diagonal and the diagonal tiles' log-determinants (summed in tile order)
static int n2ll_tiled(cocons_ctx* c, const double* theta6, const double* limits, const double* mean_p, double* logdet,
                      double* quad) {
  if (!theta6 || !limits || !logdet || !quad || c->r <= 0) {
    set_error("n2ll_taper: bad argument");
    return COCONS_ERR_ARG;
  }
  cudaSetDevice(c->device);
  int rc = assemble_and_factor(c, COCONS_PAR_DIFF, theta6, limits, mean_p, true);
  if (rc) return rc;
  cudaStream_t st = c->stream;
  std::vector<double> part((size_t)c->T), g((size_t)kTile * c->r);
  COCONS_CUDA_TRY(cudaMemcpyAsync(part.data(), c->dLogPart, sizeof(double) * c->T, cudaMemcpyDeviceToHost, st));
  COCONS_CUDA_TRY(cudaMemcpyAsync(g.data(), c->dPool + c->g_off, sizeof(double) * g.size(), cudaMemcpyDeviceToHost,
                                  st));
  COCONS_CUDA_TRY(cudaMemcpyAsync(c->hInfo, c->ws.info, sizeof(int), cudaMemcpyDeviceToHost, st));
  COCONS_CUDA_TRY(cudaEventRecord(c->ev[3], st));
  COCONS_CUDA_TRY(cudaStreamSynchronize(st));
  finish_timings(c);
  if (*c->hInfo != 0) return *c->hInfo;  // > 0: not positive definite
  double ld = 0.0;
  for (double v : part) ld += v;
  *logdet = ld;
  for (int64_t j = 0; j < c->r; ++j) quad[j] = -g[(size_t)(j * kTile + j)];
  c->factor_valid = true;
  return 0;
}

int cocons_n2ll_taper(cocons_ctx* c, const double* theta6, const double* limits, const double* mean_p,
                      double* logdet, double* quad) {
  if (!c || !c->dTap) {
    set_error("n2ll_taper: cocons_ctx_set_taper first");
    return COCONS_ERR_STATE;
  }
  if (c->tiled) return n2ll_tiled(c, theta6, limits, mean_p, logdet, quad);
  return n2ll_impl(c, COCONS_ML, theta6, limits, mean_p, logdet, quad, nullptr, nullptr, true);
}

// entry vectors of the stateless builders: rows x cols pattern, one launch
static int taper_entries_host(const char* who, int64_t n, int64_t m, int64_t p, const double* locs,
                              const double* locs_rows, const double* X, const double* X_rows, const double* theta6,
                              const double* limits, const int32_t* colindices, const int32_t* rowpointers, int64_t nnz,
                              double* out) {
  // m == 0: square pattern over the n sites (cov_rns_taper); m > 0: m prediction rows x n columns
  const bool square = (m == 0);
  const int64_t nrows = square ? n : m;
  if (n <= 0 || m < 0 || p <= 0 || !locs || !X || !theta6 || !limits || !out || (!square && (!locs_rows || !X_rows))) {
    set_error("%s: bad argument", who);
    return COCONS_ERR_ARG;
  }
  int rc = check_pattern(who, colindices, rowpointers, nrows, n, nnz);
  if (rc) return rc;
  if ((rc = check_device(default_device()))) return rc;
  double nu_fixed = 0.0;
  // the prediction variant has no fixed-smoothness shortcut (src/cocons_taper.cpp:54-70): always the Bessel branch
  const int mode = square ? smooth_mode_for(COCONS_PAR_DIFF, (int)p, theta6, limits, &nu_fixed) : (int)SM_GENERAL;
  cudaStream_t st = nullptr;
  double *dX = nullptr, *dL = nullptr, *dXr = nullptr, *dLr = nullptr, *dT = nullptr, *dS = nullptr, *dSr = nullptr,
         *dOut = nullptr;
  int *dCol = nullptr, *dRow = nullptr;
  auto cleanup = [&]() {
    cudaFree(dX), cudaFree(dL), cudaFree(dXr), cudaFree(dLr), cudaFree(dT), cudaFree(dS), cudaFree(dSr), cudaFree(dOut);
    cudaFree(dCol), cudaFree(dRow);
  };
  const int64_t nz = std::max<int64_t>(nnz, 1);
  TRY_OR_CLEAN(cudaMalloc(&dX, sizeof(double) * n * p));
  TRY_OR_CLEAN(cudaMalloc(&dL, sizeof(double) * n * 2));
  TRY_OR_CLEAN(cudaMalloc(&dT, sizeof(double) * 6 * p));
  TRY_OR_CLEAN(cudaMalloc(&dS, sizeof(double) * TF_COUNT * n));
  TRY_OR_CLEAN(cudaMalloc(&dOut, sizeof(double) * nz));
  TRY_OR_CLEAN(cudaMalloc(&dCol, sizeof(int) * nz));
  TRY_OR_CLEAN(cudaMalloc(&dRow, sizeof(int) * (nrows + 1)));
  TRY_OR_CLEAN(cudaMemcpyAsync(dX, X, sizeof(double) * n * p, cudaMemcpyHostToDevice, st));
  TRY_OR_CLEAN(cudaMemcpyAsync(dL, locs, sizeof(double) * n * 2, cudaMemcpyHostToDevice, st));
  TRY_OR_CLEAN(cudaMemcpyAsync(dT, theta6, sizeof(double) * 6 * p, cudaMemcpyHostToDevice, st));
  TRY_OR_CLEAN(cudaMemcpyAsync(dCol, colindices, sizeof(int) * nnz, cudaMemcpyHostToDevice, st));
  TRY_OR_CLEAN(cudaMemcpyAsync(dRow, rowpointers, sizeof(int) * (nrows + 1), cudaMemcpyHostToDevice, st));
  TaperTable C{dS, n}, R{dS, n};
  launch_taper_site_stage(n, (int)p, dX, n, dL, n, dT, limits[0], limits[1], mode, 0, C, st);
  if (!square) {
    TRY_OR_CLEAN(cudaMalloc(&dXr, sizeof(double) * m * p));
    TRY_OR_CLEAN(cudaMalloc(&dLr, sizeof(double) * m * 2));
    TRY_OR_CLEAN(cudaMalloc(&dSr, sizeof(double) * TF_COUNT * m));
    TRY_OR_CLEAN(cudaMemcpyAsync(dXr, X_rows, sizeof(double) * m * p, cudaMemcpyHostToDevice, st));
    TRY_OR_CLEAN(cudaMemcpyAsync(dLr, locs_rows, sizeof(double) * m * 2, cudaMemcpyHostToDevice, st));
    R = TaperTable{dSr, m};
    launch_taper_site_stage(m, (int)p, dXr, m, dLr, m, dT, limits[0], limits[1], mode, 1, R, st);
  }
  launch_taper_entries(0, nnz, nrows, dCol, dRow, R, C, square ? 1 : 0, mode, nu_fixed,
                       TaperSink{TS_VECTOR, dOut, nullptr, nullptr, nullptr, 0, 0}, st);
  TRY_OR_CLEAN(cudaGetLastError());
  TRY_OR_CLEAN(cudaMemcpyAsync(out, dOut, sizeof(double) * nnz, cudaMemcpyDeviceToHost, st));
  TRY_OR_CLEAN(cudaStreamSynchronize(st));
  cleanup();
  return 0;
}

int cocons_cov_rns_taper(int64_t n, int64_t p, const double* locs, const double* X, const double* theta6,
                         const double* smooth_limits, const int32_t* colindices, const int32_t* rowpointers,
                         int64_t nnz, double* out) {
  return taper_entries_host("cov_rns_taper", n, 0, p, locs, nullptr, X, nullptr, theta6, smooth_limits, colindices,
                            rowpointers, nnz, out);
}

int cocons_cov_rns_taper_pred(int64_t n, int64_t m, int64_t p, const double* locs, const double* locs_pred,
                              const double* X, const double* X_pred, const double* theta6,
                              const double* smooth_limits, const int32_t* colindices, const int32_t* rowpointers,
                              int64_t nnz, double* out) {
  if (m <= 0) {
    set_error("cov_rns_taper_pred: bad argument");
    return COCONS_ERR_ARG;
  }
  return taper_entries_host("cov_rns_taper_pred", n, m, p, locs, locs_pred, X, X_pred, theta6, smooth_limits,
                            colindices, rowpointers, nnz, out);
}

int cocons_profile_betas(cocons_ctx* c, int kind, double* betas) {
  if (int rc_ = refuse_tiled(c, "profile_betas")) return rc_;
  if (!c || !betas || (kind != COCONS_PROFILE && kind != COCONS_REML)) {
    set_error("profile_betas: bad argument");
    return COCONS_ERR_ARG;
  }
  if (!c->factor_valid) {
    set_error("profile_betas: no factor kept (call cocons_n2ll or cocons_factor first)");
    return COCONS_ERR_STATE;
  }
  cudaSetDevice(c->device);
  const int64_t np = c->n_pad;
  const int qx = (kind == COCONS_PROFILE) ? (int)c->q : (int)c->p;
  if (qx <= 0 || qx >= kMaxRhs) {
    set_error("profile_betas: mean design missing");
    return COCONS_ERR_STATE;
  }
  cudaStream_t st = c->stream;
  const double* src = (kind == COCONS_PROFILE) ? c->dXb : c->dX;
  COCONS_CUDA_TRY(cudaMemcpyAsync(c->dRhs, src, sizeof(double) * np * qx, cudaMemcpyDeviceToDevice, st));
  forward_solve_ws(c->dA, np, np, c->ws, c->dRhs, np, qx, st);
  // rowSums(z)/r as one right-hand side (R/optim.R:341)
  std::vector<double> zsum((size_t)np, 0.0), hz((size_t)np * c->r);
  COCONS_CUDA_TRY(cudaMemcpyAsync(hz.data(), c->dZ, sizeof(double) * np * c->r, cudaMemcpyDeviceToHost, st));
  COCONS_CUDA_TRY(cudaStreamSynchronize(st));
  for (int64_t col = 0; col < c->r; ++col)
    for (int64_t i = 0; i < c->n; ++i) zsum[(size_t)i] += hz[(size_t)col * np + i];
  double* rhs = c->dRhs + (int64_t)qx * np;
  COCONS_CUDA_TRY(cudaMemcpyAsync(rhs, zsum.data(), sizeof(double) * np, cudaMemcpyHostToDevice, st));
  forward_solve_ws(c->dA, np, np, c->ws, rhs, np, 1, st);
  const int k = qx + 1;
  launch_gram(c->dRhs, c->n, np, k, c->dGram, st);
  double* hG = c->hStage + 7 * c->p;
  COCONS_CUDA_TRY(cudaMemcpyAsync(hG, c->dGram, sizeof(double) * k * k, cudaMemcpyDeviceToHost, st));
  int rc = solve_status(c, "profile_betas");
  if (rc) return rc;
  std::vector<double> W((size_t)qx * qx);
  for (int a = 0; a < qx; ++a)
    for (int b = 0; b < qx; ++b) W[(size_t)a * qx + b] = hG[a * k + b];
  if (!small_chol(W, qx)) {
    set_error("profile_betas: X' Sigma^-1 X is not positive definite");
    return COCONS_ERR_STATE;
  }
  std::vector<double> t(qx);
  for (int a = 0; a < qx; ++a) {
    double s = hG[a * k + qx];
    for (int b = 0; b < a; ++b) s -= W[(size_t)a * qx + b] * t[b];
    t[a] = s / W[(size_t)a * qx + a];
  }
  for (int a = qx - 1; a >= 0; --a) {
    double s = t[a];
    for (int b = a + 1; b < qx; ++b) s -= W[(size_t)b * qx + a] * betas[b];
    betas[a] = s / W[(size_t)a * qx + a];
  }
  for (int a = 0; a < qx; ++a) betas[a] /= (double)c->r;
  return 0;
}

int cocons_factor(cocons_ctx* c, int par, const double* theta6, const double* limits) {
  if (int rc_ = refuse_tiled(c, "factor")) return rc_;
  if (!c || !theta6 || (par != COCONS_PAR_DIFF && par != COCONS_PAR_CLASSIC) || (par == COCONS_PAR_DIFF && !limits)) {
    set_error("factor: bad argument");
    return COCONS_ERR_ARG;
  }
  cudaSetDevice(c->device);
  int rc = assemble_and_factor(c, par, theta6, limits, nullptr);
  if (rc) return rc;
  COCONS_CUDA_TRY(cudaEventRecord(c->ev[3], c->stream));
  COCONS_CUDA_TRY(cudaMemcpyAsync(c->hInfo, c->ws.info, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  COCONS_CUDA_TRY(cudaStreamSynchronize(c->stream));
  finish_timings(c);
  if (*c->hInfo != 0) return *c->hInfo;
  c->factor_valid = true;
  return 0;
}

// T = C L^-T for a block of prediction sites, in place on dC (mp x n_pad, ld = mp), right-looking with the
// same two-level blocking as the factorisation: inside a 512-wide panel, column tile J gets
// T_J = C_J inv(L_JJ)^T and updates the rest of the panel (K = 128); the columns right of the panel are then
// updated once with K = 512, which is where the flops are.
static void right_solve_lt(cocons_ctx* c, double* dC, int64_t mp) {
  static int outer_env = -1;
  if (outer_env < 0) { const char* e = getenv("COCONS_PRED_OUTER"); outer_env = e ? atoi(e) : 4; }
  const int64_t np = c->n_pad, nt = np / kTile, outer = outer_env;
  for (int64_t J0 = 0; J0 < nt; J0 += outer) {
    const int64_t jb = std::min<int64_t>(outer, nt - J0);
    for (int64_t J = J0; J < J0 + jb; ++J) {
      double* CJ = dC + J * kTile * mp;
      launch_gemm_nt(1, mp, kTile, kTile, CJ, mp, c->ws.winv + J * (int64_t)kTile * kTile, kTile, CJ, mp, 0,
                     c->stream);
      const int64_t rest = (J0 + jb - J - 1) * kTile;  // remaining columns of this panel
      if (rest > 0)
        launch_gemm_nt(0, mp, rest, kTile, CJ, mp, c->dA + J * kTile * np + (J + 1) * kTile, np, CJ + kTile * mp, mp,
                       0, c->stream);
    }
    const int64_t done = (J0 + jb) * kTile, trail = np - done;
    if (trail > 0)  // C[:, done:] -= T[:, panel] L[done:, panel]^T
      launch_gemm_nt(0, mp, trail, jb * kTile, dC + J0 * kTile * mp, mp, c->dA + J0 * kTile * np + done, np,
                     dC + done * mp, mp, 0, c->stream);
  }
}

struct PredBlock {
  double *dXp = nullptr, *dLp = nullptr, *dSp = nullptr, *dC = nullptr;
  ~PredBlock() { cudaFree(dXp), cudaFree(dLp), cudaFree(dSp), cudaFree(dC); }
};

// the prediction pattern of the tapered model (pred_taper, R/predict.R:233-249): m rows x n columns
struct TaperPred {
  const int32_t* rowpointers = nullptr;  // host, 1-based
  int *dCol = nullptr, *dRow = nullptr;
  double* dTap = nullptr;
  ~TaperPred() { cudaFree(dCol), cudaFree(dRow), cudaFree(dTap); }
};

// builds T = C L^-T for prediction sites [i0, i0+mc) into blk.dC (mp x n_pad)
static int pred_block(cocons_ctx* c, PredBlock& blk, int64_t m, int64_t i0, int64_t mc, int64_t mp,
                      const double* locs_pred, const double* Xp, const TaperPred* tp) {
  const int64_t np = c->n_pad, p = c->p;
  std::vector<double> hx((size_t)mp * p, 0.0), hl((size_t)mp * 2, 0.0);
  for (int64_t k = 0; k < p; ++k)
    for (int64_t i = 0; i < mc; ++i) hx[(size_t)k * mp + i] = Xp[(size_t)k * m + i0 + i];
  for (int64_t k = 0; k < 2; ++k)
    for (int64_t i = 0; i < mc; ++i) hl[(size_t)k * mp + i] = locs_pred[(size_t)k * m + i0 + i];
  cudaStream_t st = c->stream;
  COCONS_CUDA_TRY(cudaMemcpyAsync(blk.dXp, hx.data(), sizeof(double) * hx.size(), cudaMemcpyHostToDevice, st));
  COCONS_CUDA_TRY(cudaMemcpyAsync(blk.dLp, hl.data(), sizeof(double) * hl.size(), cudaMemcpyHostToDevice, st));
  COCONS_CUDA_TRY(cudaMemsetAsync(blk.dC, 0, sizeof(double) * mp * np, st));
  if (tp) {
    // taper * cov_rns_taper_pred on the rows of this block (src/cocons_taper.cpp:17-139)
    TaperTable P{blk.dSp, mp};
    launch_taper_site_stage(mc, (int)p, blk.dXp, mp, blk.dLp, mp, c->dTheta, c->lim[0], c->lim[1], SM_GENERAL, 1, P, st);
    const int64_t e0 = (int64_t)tp->rowpointers[i0] - 1, e1 = (int64_t)tp->rowpointers[i0 + mc] - 1;
    launch_taper_entries(e0, e1 - e0, m, tp->dCol, tp->dRow, P, c->taper_table(), 0, SM_GENERAL, 0.0,
                         TaperSink{TS_ROWS, nullptr, tp->dTap, c->dInv, blk.dC, mp, i0}, st);
  } else {
    SiteTable P{blk.dSp, mp, nullptr};
    // cov_rns_pred always evaluates smoothness through the logistic (src/cocons_full.cpp:381,401)
    const int pmode = (c->mode == SM_CLASSIC) ? SM_CLASSIC : SM_GENERAL;
    launch_site_stage(mc, mp, (int)p, blk.dXp, mp, blk.dLp, mp, c->dTheta, c->lim[0], c->lim[1], pmode, P, st);
    // the training table was built for cov_rns; its smooth column is only valid in general mode
    launch_assemble_cross(mc, c->n, P, c->table(), c->global_range, blk.dC, mp, st);
  }
  COCONS_CUDA_TRY(cudaStreamSynchronize(st));  // hx/hl go out of scope
  right_solve_lt(c, blk.dC, mp);
  COCONS_CUDA_TRY(cudaGetLastError());
  return 0;
}

// the training site table must carry logistic smoothness for the cross-covariance
static int refresh_table_for_pred(cocons_ctx* c) {
  if (c->mode == SM_GENERAL || c->mode == SM_CLASSIC) return 0;
  launch_site_stage(c->n, c->n_pad, (int)c->p, c->dX, c->n_pad, c->dLocs, c->n_pad, c->dTheta, c->lim[0], c->lim[1],
                    SM_GENERAL, c->table(), c->stream);
  COCONS_CUDA_TRY(cudaGetLastError());
  return 0;
}

static int predict_impl(cocons_ctx* c, int64_t m, const double* locs_pred, const double* Xp, const double* resid,
                        double* stochastic, double* explained, const TaperPred* tp) {
  if (int rc_ = refuse_tiled(c, "predict")) return rc_;
  if (!c || m <= 0 || !locs_pred || !Xp || !resid || !stochastic) {
    set_error("predict: bad argument");
    return COCONS_ERR_ARG;
  }
  if (!c->factor_valid) {
    set_error("predict: no factor kept (call cocons_factor first)");
    return COCONS_ERR_STATE;
  }
  if (c->mode == SM_CLASSIC) {
    set_error("predict: the kept factor uses the classic parameterisation; cocoPredict is 'diff' only");
    return COCONS_ERR_STATE;
  }
  if (c->factor_is_taper != (tp != nullptr)) {
    set_error(tp ? "predict_taper: the kept factor is of the dense model (call cocons_factor_taper first)"
                 : "predict: the kept factor is of the tapered model; use cocons_predict_taper");
    return COCONS_ERR_STATE;
  }
  cudaSetDevice(c->device);
  int rc = 0;
  if (tp) {
    // cov_rns_taper_pred always takes the smoothness through the logistic, for both site sets (:54-70)
    launch_taper_site_stage(c->n, (int)c->p, c->dX, c->n_pad, c->dLocs, c->n_pad, c->dTheta, c->lim[0], c->lim[1],
                            SM_GENERAL, 0, c->taper_table(), c->stream);
  } else if ((rc = refresh_table_for_pred(c))) {
    return rc;
  }
  const int64_t np = c->n_pad, p = c->p;
  cudaStream_t st = c->stream;
  // y = L^-1 resid (sorted order)
  {
    std::vector<double> hr((size_t)np, 0.0);
    for (int64_t s = 0; s < c->n; ++s) hr[(size_t)s] = resid[c->perm[(size_t)s]];
    COCONS_CUDA_TRY(cudaMemcpyAsync(c->dRhs, hr.data(), sizeof(double) * np, cudaMemcpyHostToDevice, st));
    COCONS_CUDA_TRY(cudaStreamSynchronize(st));
    forward_solve_ws(c->dA, np, np, c->ws, c->dRhs, np, 1, st);
  }
  const int64_t mc_max = std::min<int64_t>(round_up(m, kTile), 4096);
  PredBlock blk;
  COCONS_CUDA_TRY(cudaMalloc(&blk.dXp, sizeof(double) * mc_max * p));
  COCONS_CUDA_TRY(cudaMalloc(&blk.dLp, sizeof(double) * mc_max * 2));
  COCONS_CUDA_TRY(cudaMalloc(&blk.dSp, sizeof(double) * SF_COUNT * mc_max));
  COCONS_CUDA_TRY(cudaMalloc(&blk.dC, sizeof(double) * mc_max * np));
  const int nsl = 16;
  double* dPart = nullptr;
  COCONS_CUDA_TRY(cudaMalloc(&dPart, sizeof(double) * 2 * nsl * mc_max));
  std::vector<double> hp((size_t)2 * nsl * mc_max);
  for (int64_t i0 = 0; i0 < m; i0 += mc_max) {
    const int64_t mc = std::min<int64_t>(mc_max, m - i0), mp = mc_max;
    if ((rc = pred_block(c, blk, m, i0, mc, mp, locs_pred, Xp, tp))) {
      cudaFree(dPart);
      return rc;
    }
    note_launch();
    pred_reduce_kernel<<<dim3((unsigned)((mc + 127) / 128), nsl), 128, 0, st>>>(blk.dC, mp, mc, c->n, c->dRhs, nsl,
                                                                                dPart, dPart + nsl * mc_max);
    cudaError_t e = cudaMemcpyAsync(hp.data(), dPart, sizeof(double) * 2 * nsl * mc_max, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
      set_error("predict: %s", cudaGetErrorString(e));
      cudaFree(dPart);
      return COCONS_ERR_CUDA;
    }
    for (int64_t i = 0; i < mc; ++i) {
      double a = 0, b = 0;
      for (int s = 0; s < nsl; ++s) {
        a += hp[(size_t)s * mc + i];
        b += hp[(size_t)(nsl * mc_max) + (size_t)s * mc + i];
      }
      stochastic[i0 + i] = a;
      if (explained) explained[i0 + i] = b;
    }
  }
  cudaFree(dPart);
  return solve_status(c, "predict");
}

int cocons_predict(cocons_ctx* c, int64_t m, const double* locs_pred, const double* Xp, const double* resid,
                   double* stochastic, double* explained) {
  return predict_impl(c, m, locs_pred, Xp, resid, stochastic, explained, nullptr);
}

int cocons_factor_taper(cocons_ctx* c, const double* theta6, const double* limits) {
  if (!c || !theta6 || !limits) {
    set_error("factor_taper: bad argument");
    return COCONS_ERR_ARG;
  }
  if (!c->dTap) {
    set_error("factor_taper: cocons_ctx_set_taper first");
    return COCONS_ERR_STATE;
  }
  cudaSetDevice(c->device);
  int rc = assemble_and_factor(c, COCONS_PAR_DIFF, theta6, limits, nullptr, true);
  if (rc) return rc;
  COCONS_CUDA_TRY(cudaEventRecord(c->ev[3], c->stream));
  COCONS_CUDA_TRY(cudaMemcpyAsync(c->hInfo, c->ws.info, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  COCONS_CUDA_TRY(cudaStreamSynchronize(c->stream));
  finish_timings(c);
  if (*c->hInfo != 0) return *c->hInfo;
  c->factor_valid = true;
  return 0;
}

int cocons_predict_taper(cocons_ctx* c, int64_t m, const double* locs_pred, const double* Xp,
                         const int32_t* colindices, const int32_t* rowpointers, const double* taper_entries,
                         int64_t nnz, const double* resid, double* stochastic, double* explained) {
  if (int rc_ = refuse_tiled(c, "predict_taper")) return rc_;
  if (!c || m <= 0 || !taper_entries) {
    set_error("predict_taper: bad argument");
    return COCONS_ERR_ARG;
  }
  int rc = check_pattern("predict_taper", colindices, rowpointers, m, c->n, nnz);
  if (rc) return rc;
  cudaSetDevice(c->device);
  TaperPred tp;
  tp.rowpointers = rowpointers;
  const int64_t nz = std::max<int64_t>(nnz, 1);
  COCONS_CUDA_TRY(cudaMalloc(&tp.dCol, sizeof(int) * nz));
  COCONS_CUDA_TRY(cudaMalloc(&tp.dRow, sizeof(int) * (m + 1)));
  COCONS_CUDA_TRY(cudaMalloc(&tp.dTap, sizeof(double) * nz));
  COCONS_CUDA_TRY(cudaMemcpy(tp.dCol, colindices, sizeof(int) * nnz, cudaMemcpyHostToDevice));
  COCONS_CUDA_TRY(cudaMemcpy(tp.dRow, rowpointers, sizeof(int) * (m + 1), cudaMemcpyHostToDevice));
  COCONS_CUDA_TRY(cudaMemcpy(tp.dTap, taper_entries, sizeof(double) * nnz, cudaMemcpyHostToDevice));
  return predict_impl(c, m, locs_pred, Xp, resid, stochastic, explained, &tp);
}

int cocons_sim(cocons_ctx* c, int64_t k, const double* eps, double* out) {
  if (int rc_ = refuse_tiled(c, "sim")) return rc_;
  if (!c || k <= 0 || !eps || !out) {
    set_error("sim: bad argument");
    return COCONS_ERR_ARG;
  }
  if (!c->factor_valid) {
    set_error("sim: no factor kept (call cocons_factor first)");
    return COCONS_ERR_STATE;
  }
  cudaSetDevice(c->device);
  const int64_t np = c->n_pad;
  cudaStream_t st = c->stream;
  double *dE = nullptr, *dO = nullptr;
  COCONS_CUDA_TRY(cudaMalloc(&dE, sizeof(double) * np * k));
  if (cudaMalloc(&dO, sizeof(double) * np * k) != cudaSuccess) {
    cudaFree(dE);
    set_error("sim: out of device memory");
    return COCONS_ERR_ALLOC;
  }
  std::vector<double> h((size_t)np * k, 0.0);
  for (int64_t col = 0; col < k; ++col)
    for (int64_t s = 0; s < c->n; ++s) h[(size_t)col * np + s] = eps[(size_t)col * c->n + c->perm[(size_t)s]];
  cudaError_t e = cudaMemcpyAsync(dE, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    launch_trmm_lower(c->dA, np, np, dE, dO, np, (int)k, st);
    e = cudaMemcpyAsync(h.data(), dO, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, st);
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(dE), cudaFree(dO);
  if (e != cudaSuccess) {
    set_error("sim: %s", cudaGetErrorString(e));
    return COCONS_ERR_CUDA;
  }
  for (int64_t col = 0; col < k; ++col)
    for (int64_t s = 0; s < c->n; ++s) out[(size_t)col * c->n + c->perm[(size_t)s]] = h[(size_t)col * np + s];
  return 0;
}

int cocons_sim_cond(cocons_ctx* c, int64_t m, const double* locs_pred, const double* Xp, int64_t k, const double* eps,
                    double* out) {
  if (int rc_ = refuse_tiled(c, "sim_cond")) return rc_;
  if (!c || m <= 0 || k <= 0 || !locs_pred || !Xp || !eps || !out) {
    set_error("sim_cond: bad argument");
    return COCONS_ERR_ARG;
  }
  if (!c->factor_valid) {
    set_error("sim_cond: no factor kept (call cocons_factor first)");
    return COCONS_ERR_STATE;
  }
  if (c->mode == SM_CLASSIC) {
    set_error("sim_cond: the reference's conditional branch uses the 'diff' parameterisation only");
    return COCONS_ERR_ARG;
  }
  if (c->factor_is_taper) {
    set_error("sim_cond: the reference's conditional branch is dense-only (R/sim.R:69-121)");
    return COCONS_ERR_STATE;
  }
  cudaSetDevice(c->device);
  const int64_t np = c->n_pad, p = c->p, mp = round_up(m, kTile);
  cudaStream_t st = c->stream;
  // covmat_unobs = cov_rns(theta, locs_pred, X_pred, limits) with the factor's own mode (R/sim.R:99-102)
  const int own_mode = c->mode;
  int rc = refresh_table_for_pred(c);
  if (rc) return rc;
  PredBlock blk;
  double *dS = nullptr, *dE = nullptr, *dO = nullptr;
  CholWorkspace ws2{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  auto cleanup = [&]() { cudaFree(dS), cudaFree(dE), cudaFree(dO), chol_workspace_destroy(&ws2); };
  if (cudaMalloc(&blk.dXp, sizeof(double) * mp * p) != cudaSuccess ||
      cudaMalloc(&blk.dLp, sizeof(double) * mp * 2) != cudaSuccess ||
      cudaMalloc(&blk.dSp, sizeof(double) * SF_COUNT * mp) != cudaSuccess ||
      cudaMalloc(&blk.dC, sizeof(double) * mp * np) != cudaSuccess ||
      cudaMalloc(&dS, sizeof(double) * mp * mp) != cudaSuccess || cudaMalloc(&dE, sizeof(double) * mp * k) != cudaSuccess ||
      cudaMalloc(&dO, sizeof(double) * mp * k) != cudaSuccess ||
      chol_workspace_create(mp, &ws2, true) != 0) {
    cleanup();
    set_error("sim_cond: out of device memory");
    return COCONS_ERR_ALLOC;
  }
  if ((rc = pred_block(c, blk, m, 0, m, mp, locs_pred, Xp, nullptr))) {
    cleanup();
    return rc;
  }
  // S_pp on the prediction sites, with the smoothness handling of cov_rns itself
  SiteTable P{blk.dSp, mp, nullptr};
  launch_site_stage(m, mp, (int)p, blk.dXp, mp, blk.dLp, mp, c->dTheta, c->lim[0], c->lim[1], own_mode, P, st);
  launch_assemble_lower(m, mp, P, c->global_range, c->nu_fixed, own_mode, dS, mp, st);
  // Schur complement: S_pp - T T^T, T = C L^-T (R/sim.R:106)
  launch_gemm_nt(0, mp, mp, np, blk.dC, mp, blk.dC, mp, dS, mp, 1, st);
  chol_factor(dS, mp, mp, ws2, st);
  std::vector<double> h((size_t)mp * k, 0.0);
  for (int64_t col = 0; col < k; ++col)
    for (int64_t i = 0; i < m; ++i) h[(size_t)col * mp + i] = eps[(size_t)col * m + i];
  int info = 0;
  cudaError_t e = cudaMemcpyAsync(dE, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    launch_trmm_lower(dS, mp, mp, dE, dO, mp, (int)k, st);
    e = cudaMemcpyAsync(h.data(), dO, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, st);
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(&info, ws2.info, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cleanup();
  if (e != cudaSuccess) {
    set_error("sim_cond: %s", cudaGetErrorString(e));
    return COCONS_ERR_CUDA;
  }
  if (info != 0) return info;
  for (int64_t col = 0; col < k; ++col)
    for (int64_t i = 0; i < m; ++i) out[(size_t)col * m + i] = h[(size_t)col * mp + i];
  return 0;
}

int cocons_ctx_get_factor(cocons_ctx* c, double* L, int64_t* perm) {
  if (!c || !L) {
    set_error("get_factor: bad argument");
    return COCONS_ERR_ARG;
  }
  if (!c->factor_valid) {
    set_error("get_factor: no factor kept");
    return COCONS_ERR_STATE;
  }
  cudaSetDevice(c->device);
  const int64_t np = c->n_pad, n = c->n;
  if (c->tiled) {  // expand the stored tiles (meant for small n: the whole pool goes through the host)
    std::vector<double> pool((size_t)c->pool_elems);
    COCONS_CUDA_TRY(cudaMemcpy(pool.data(), c->dPool, sizeof(double) * pool.size(), cudaMemcpyDeviceToHost));
    std::fill(L, L + (size_t)n * n, 0.0);
    for (int64_t J = 0; J < c->T; ++J)
      for (int64_t k = c->colptr[(size_t)J]; k < c->colptr[(size_t)J + 1]; ++k) {
        const int64_t I = c->rows[(size_t)k];
        const double* t = pool.data() + c->base[(size_t)J] + (k - c->colptr[(size_t)J]) * kTile;
        for (int64_t jj = 0; jj < kTile && J * kTile + jj < n; ++jj)
          for (int64_t ii = 0; ii < kTile && I * kTile + ii < n; ++ii)
            if (I * kTile + ii >= J * kTile + jj)
              L[(size_t)(J * kTile + jj) * n + I * kTile + ii] = t[jj * c->ldp[(size_t)J] + ii];
      }
    if (perm)
      for (int64_t s = 0; s < n; ++s) perm[s] = c->perm[(size_t)s];
    return 0;
  }
  COCONS_CUDA_TRY(cudaMemcpy2D(L, sizeof(double) * n, c->dA, sizeof(double) * np, sizeof(double) * n, n,
                               cudaMemcpyDeviceToHost));
  for (int64_t j = 0; j < n; ++j)
    for (int64_t i = 0; i < j; ++i) L[(size_t)j * n + i] = 0.0;
  if (perm)
    for (int64_t s = 0; s < n; ++s) perm[s] = c->perm[(size_t)s];
  return 0;
}

int cocons_ctx_factor_rows(cocons_ctx* c, const int64_t* sites, int64_t m, double* rows, int64_t* pos) {
  if (!c || !sites || !rows || !pos || m <= 0) {
    set_error("factor_rows: bad argument");
    return COCONS_ERR_ARG;
  }
  if (!c->factor_valid) {
    set_error("factor_rows: no factor kept");
    return COCONS_ERR_STATE;
  }
  cudaSetDevice(c->device);
  const int64_t np = c->n_pad, n = c->n;
  std::vector<int64_t> inv((size_t)n);
  for (int64_t s = 0; s < n; ++s) inv[(size_t)c->perm[(size_t)s]] = s;
  for (int64_t a = 0; a < m; ++a) {
    if (sites[a] < 0 || sites[a] >= n) {
      set_error("factor_rows: site %lld out of range", (long long)sites[a]);
      return COCONS_ERR_ARG;
    }
    const int64_t i = inv[(size_t)sites[a]];
    pos[a] = i;
    double* out = rows + (size_t)a * n;
    if (c->tiled) {  // row i crosses the stored tiles (I, J) of its tile row, J <= I
      const int64_t I = i / kTile;
      std::fill(out, out + n, 0.0);
      for (int64_t J = 0; J <= I; ++J) {
        const int64_t pos = tile_pos(c, I, J);
        if (pos < 0) continue;
        const int64_t w = std::min<int64_t>(kTile, std::min(i + 1, n) - J * kTile);
        COCONS_CUDA_TRY(cudaMemcpy2D(out + J * kTile, sizeof(double), c->dPool + c->base[(size_t)J] + pos * kTile + i % kTile,
                                     sizeof(double) * c->ldp[(size_t)J], sizeof(double), (size_t)w,
                                     cudaMemcpyDeviceToHost));
      }
      continue;
    }
    // row i of the column-major factor: one element per column, columns 0..i
    COCONS_CUDA_TRY(cudaMemcpy2D(out, sizeof(double), c->dA + i, sizeof(double) * np, sizeof(double), (size_t)(i + 1),
                                 cudaMemcpyDeviceToHost));
    for (int64_t k = i + 1; k < n; ++k) out[k] = 0.0;
  }
  return 0;
}

int64_t cocons_debug_solve_units(int64_t n_pad, int32_t* units4, int64_t capacity) {
  if (n_pad <= 0 || n_pad % kTile) return COCONS_ERR_ARG;
  std::vector<int> u;
  const int64_t count = build_solve_units(n_pad / kTile, &u);
  if (units4)
    for (int64_t i = 0; i < 4 * count && i < 4 * capacity; ++i) units4[i] = u[(size_t)i];
  return count;
}

int cocons_ctx_dims(cocons_ctx* c, int64_t* dims4) {
  if (!c || !dims4) return COCONS_ERR_ARG;
  dims4[0] = c->n, dims4[1] = c->p, dims4[2] = c->r, dims4[3] = c->q;
  return 0;
}

int cocons_ctx_timings(cocons_ctx* c, double* ms4) {
  if (!c || !ms4) return COCONS_ERR_ARG;
  for (int i = 0; i < 4; ++i) ms4[i] = c->ms[i];
  return 0;
}

int cocons_ctx_debug_checksums(cocons_ctx* c, double* out2) {
  if (int rc_ = refuse_tiled(c, "ctx_debug_checksums")) return rc_;
  if (!c || !out2) return COCONS_ERR_ARG;
  out2[0] = c->check[0], out2[1] = c->check[1];
  return 0;
}

int cocons_ctx_kernel_timing(cocons_ctx* c, double* ms, double* flops) {
  if (int rc_ = refuse_tiled(c, "ctx_kernel_timing")) return rc_;
  if (!c || !ms || !flops) return COCONS_ERR_ARG;
  *ms = c->kernel_ms, *flops = c->kernel_flops;
  return 0;
}

// ---- one-shot objective ----------------------------------------------------

static std::mutex g_ws_mutex;
static cocons_ctx* g_ws = nullptr;

void cocons_release_workspace(void) {
  std::lock_guard<std::mutex> lock(g_ws_mutex);
  if (g_ws) cocons_ctx_destroy(g_ws), g_ws = nullptr;
}

int cocons_neg2loglik_dense(int kind, int64_t n, int64_t p, int64_t r, int64_t q, const double* locs, const double* X,
                            const double* z, const double* xb, const double* theta6, const double* limits,
                            const double* mean_p, double* logdet, double* quad, double* logdet_w, int* rank_x) {
  std::lock_guard<std::mutex> lock(g_ws_mutex);
  const int device = default_device();
  int rc;
  if (g_ws && (g_ws->n != n || g_ws->p != p || g_ws->r != r || g_ws->device != device)) {
    cocons_ctx_destroy(g_ws);
    g_ws = nullptr;
  }
  if (!g_ws) {
    if ((rc = cocons_ctx_create(device, n, p, r, locs, X, z, nullptr, &g_ws))) return rc;
  } else {
    // same shapes: refresh the data in place (the caller hands R objects over on every call)
    cocons_ctx* c = g_ws;
    cudaSetDevice(c->device);
    morton_order(n, locs, c->perm.data());
    c->hX.assign(X, X + (size_t)n * p);
    c->rank_x = -1;
    // the inverse permutation and any attached taper pattern follow perm: drop them (a taper has to be attached
    // again after new locations; cocons_n2ll_taper reports COCONS_ERR_STATE otherwise)
    cudaFree(c->dInv), cudaFree(c->dTapCol), cudaFree(c->dTapRow), cudaFree(c->dTap);
    c->dInv = c->dTapCol = c->dTapRow = nullptr, c->dTap = nullptr, c->tap_nnz = 0;
    std::vector<int> orig((size_t)c->n_pad);
    for (int64_t s = 0; s < c->n_pad; ++s) orig[(size_t)s] = (s < n) ? (int)c->perm[(size_t)s] : (int)s;
    COCONS_CUDA_TRY(cudaMemcpy(c->dOrig, orig.data(), sizeof(int) * c->n_pad, cudaMemcpyHostToDevice));
    if ((rc = upload_sorted(c, X, p, c->dX)) || (rc = upload_sorted(c, locs, 2, c->dLocs)) ||
        (rc = upload_sorted(c, z, r, c->dZ)))
      return rc;
  }
  if (kind == COCONS_PROFILE) {
    if (!xb || q <= 0) {
      set_error("neg2loglik_dense: COCONS_PROFILE needs x_betas");
      return COCONS_ERR_ARG;
    }
    if ((rc = cocons_ctx_set_xbetas(g_ws, q, xb))) return rc;
  }
  return cocons_n2ll(g_ws, kind, theta6, limits, mean_p, logdet, quad, logdet_w, rank_x);
}

// ---- measurement helper -----------------------------------------------------

__global__ void fill_kernel(double* p, int64_t count, double scale) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) p[i] = scale * (double)(((uint64_t)i * 2654435761ull) % 1024ull) / 1024.0;
}

int cocons_bench_syrk(int device, int64_t n, int64_t k, int reps, double* ms_per_rep) {
  int rc = check_device(device);
  if (rc) return rc;
  if (n % kTile || k % 16 || !ms_per_rep || reps <= 0) {
    set_error("bench_syrk: n must be a multiple of 128 and k of 16");
    return COCONS_ERR_ARG;
  }
  double *dC = nullptr, *dP = nullptr;
  COCONS_CUDA_TRY(cudaMalloc(&dC, sizeof(double) * n * n));
  if (cudaMalloc(&dP, sizeof(double) * n * k) != cudaSuccess) {
    cudaFree(dC);
    set_error("bench_syrk: out of device memory");
    return COCONS_ERR_ALLOC;
  }
  fill_kernel<<<(unsigned)((n * n + 255) / 256), 256>>>(dC, n * n, 1.0);
  fill_kernel<<<(unsigned)((n * k + 255) / 256), 256>>>(dP, n * k, 1e-3);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0), cudaEventCreate(&e1);
  launch_gemm_nt(0, n, n, k, dP, n, dP, n, dC, n, 1, nullptr);
  cudaEventRecord(e0);
  for (int i = 0; i < reps; ++i) launch_gemm_nt(0, n, n, k, dP, n, dP, n, dC, n, 1, nullptr);
  cudaEventRecord(e1);
  cudaError_t e = cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0), cudaEventDestroy(e1);
  cudaFree(dC), cudaFree(dP);
  if (e != cudaSuccess) {
    set_error("bench_syrk: %s", cudaGetErrorString(e));
    return COCONS_ERR_CUDA;
  }
  *ms_per_rep = ms / reps;
  return 0;
}

int cocons_trailing_update(int device, int64_t m, const double* P, double* C, int path, int reps, double* ms_per_rep) {
  int rc = check_device(device);
  if (rc) return rc;
  if (m <= 0 || m % kTile || (path != 0 && path != 1) || reps < 0 || (reps > 0 && !ms_per_rep) || (!P != !C)) {
    set_error("trailing_update: m must be a positive multiple of 128, path 0 or 1, and P and C both given or both "
              "null");
    return COCONS_ERR_ARG;
  }
  if (path == 1 && !g_syrk_i8.update) {
    set_error("trailing_update: this build of the library has no split-int8 update");
    return COCONS_ERR_STATE;
  }
  const int64_t k = kSyrkI8K;
  double *dC = nullptr, *dP = nullptr, *dS = nullptr;
  int8_t* dQ = nullptr;
  int* dInfo = nullptr;
  if (cudaMalloc(&dC, sizeof(double) * m * m) != cudaSuccess || cudaMalloc(&dP, sizeof(double) * m * k) != cudaSuccess ||
      (path == 1 && (cudaMalloc(&dQ, (size_t)kSyrkI8BytesPerRow * m) != cudaSuccess ||
                     cudaMalloc(&dS, sizeof(double) * m) != cudaSuccess ||
                     cudaMalloc(&dInfo, sizeof(int)) != cudaSuccess))) {
    cudaFree(dC), cudaFree(dP), cudaFree(dQ), cudaFree(dS), cudaFree(dInfo);
    set_error("trailing_update: out of device memory");
    return COCONS_ERR_ALLOC;
  }
  if (dInfo) cudaMemsetAsync(dInfo, 0, sizeof(int), nullptr);
  if (P) {
    cudaMemcpy(dP, P, sizeof(double) * m * k, cudaMemcpyHostToDevice);
    cudaMemcpy(dC, C, sizeof(double) * m * m, cudaMemcpyHostToDevice);
  } else {  // every double 0x3F3F3F3F3F3F3F3F (about 4.8e-4): the timing does not depend on the values
    cudaMemsetAsync(dC, 0x3F, sizeof(double) * m * m, nullptr);
    cudaMemsetAsync(dP, 0x3F, sizeof(double) * m * k, nullptr);
  }
  auto run = [&]() {
    if (path == 1) {
      g_syrk_i8.split(dP, m, m, dQ, dS, nullptr);
      g_syrk_i8.update(m, m, dQ, dS, 0, 0, dC, m, 1, dInfo, nullptr);
    } else {
      launch_gemm_nt(0, m, m, k, dP, m, dP, m, dC, m, 1, nullptr);
    }
  };
  run();
  if (C) cudaMemcpy(C, dC, sizeof(double) * m * m, cudaMemcpyDeviceToHost);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0), cudaEventCreate(&e1);
  cudaEventRecord(e0);
  for (int i = 0; i < reps; ++i) run();
  cudaEventRecord(e1);
  cudaError_t e = cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0), cudaEventDestroy(e1);
  int info = 0;
  if (dInfo && e == cudaSuccess) e = cudaMemcpy(&info, dInfo, sizeof(int), cudaMemcpyDeviceToHost);
  cudaFree(dC), cudaFree(dP), cudaFree(dQ), cudaFree(dS), cudaFree(dInfo);
  if (e != cudaSuccess) {
    set_error("trailing_update: %s", cudaGetErrorString(e));
    return COCONS_ERR_CUDA;
  }
  if (info != 0) {
    set_error("trailing_update: a barrier wait of the split-int8 update gave up");
    return COCONS_ERR_CUDA;
  }
  if (reps > 0) *ms_per_rep = ms / reps;
  return 0;
}

}  // extern "C"
