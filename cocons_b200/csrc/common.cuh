// Shared declarations of the cocons_b200 CUDA library (sm_100a only).
#ifndef COCONS_COMMON_CUH
#define COCONS_COMMON_CUH

#include <cuda_runtime.h>
#include <stdint.h>

namespace cocons {

constexpr int kTile = 128;  // factorisation tile edge; matrices are padded to a multiple of it

// Per-site quantities, struct-of-arrays (field f of site s at base[f*stride + s]).
// They are the hoistable, bit-identical sub-expressions of the reference's pair
// loop (SURVEY.md App. A; src/cocons_full.cpp:98-107, 260-297).
enum SiteField {
  SF_X = 0,  // locs[,1]
  SF_Y,      // locs[,2]
  SF_R,      // range_det      = E(2 scale_je)
  SF_A2,     // aniso_det^2
  SF_RA,     // range_det * aniso_det
  SF_CS,     // cos(tilt)
  SF_P22,    // rnd(r * a2)                 } the c*d product of kahan() and its
  SF_E22,    // fma(r, a2, -P22)            } rounding error, for the "jj" role
  SF_P12,    // rnd(ra * cos t)
  SF_E12,    // fma(ra, cos t, -P12)
  SF_NU,     // smooth_vector (sqrt of the logistic, or exp() for classic)
  SF_SIG,    // sigma_vector   = E(0.5 std.dev)
  SF_W,      // dets_vector * sin(tilt)
  SF_AMP,    // SF_SIG * sqrt(SF_W): the site's share of the amplitude, what the pair loop reads
  SF_DV,     // E(std.dev) + nugget  (diagonal / coincident value)
  SF_COUNT
};

struct SiteTable {
  double* base;
  int64_t stride;
  const int* orig;  // original (caller-order) index of each site, or nullptr for identity
  __host__ __device__ const double* f(int k) const { return base + (int64_t)k * stride; }
  __host__ __device__ double* fw(int k) const { return base + (int64_t)k * stride; }
};

// how nu_ij is obtained (src/cocons_full.cpp:77-96, 114, 524/554)
enum SmoothMode {
  SM_GENERAL = 0,     // nu_ij = s_i s_j, Bessel branch
  SM_HALF = 1,        // fixed nu = 0.5 closed form
  SM_THREEHALF = 2,   // fixed nu = 1.5
  SM_FIVEHALF = 3,    // fixed nu = 2.5
  SM_CLASSIC = 4,     // nu_ij = (nu_i + nu_j)/2, nu_i = exp(.)
  SM_DEGENERATE = 5   // fixed non-half-integer nu in cov_rns: smooth_vector stays 0 (SURVEY App. B-1)
};

void set_error(const char* fmt, ...);
void note_launch(int count = 1);  // kernel-launch counter behind cocons_launch_count()

#define COCONS_CUDA_TRY(expr)                                                                  \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      ::cocons::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return COCONS_ERR_CUDA;                                                                  \
    }                                                                                          \
  } while (0)

// ---- assembly.cu ---------------------------------------------------------
int smooth_mode_for(int par, int p, const double* theta6_host, const double* limits_host, double* nu_fixed);
void launch_site_stage(int64_t n, int64_t n_fill, int p, const double* dX, int64_t ldx, const double* dlocs,
                       int64_t ldl, const double* dtheta6, double lim0, double lim1, int mode, SiteTable T,
                       cudaStream_t st);
void launch_assemble_lower(int64_t n, int64_t n_out, SiteTable T, double global_range, double nu_fixed, int mode,
                           double* C, int64_t ld, cudaStream_t st);
void launch_assemble_panel(int64_t n, int64_t n_out, SiteTable T, double global_range, double nu_fixed, int mode,
                           double* slab, int64_t ld, int col_tile0, int ncol_tiles, cudaStream_t st);
void launch_assemble_cyclic(int64_t n, int64_t n_out, SiteTable T, double global_range, double nu_fixed, int mode,
                            double* slab, int64_t ld, int world, int rank, int64_t nlocal, cudaStream_t st);
void launch_assemble_cross(int64_t m, int64_t n, SiteTable Tpred, SiteTable Ttrain, double global_range, double* C,
                           int64_t ld, cudaStream_t st);
void launch_symmetrize(int64_t n, double* C, int64_t ld, cudaStream_t st);
void morton_order(int64_t n, const double* locs, int64_t* perm);

// ---- taper.cu (sparse / tapered model, src/cocons_taper.cpp) ---------------
enum TaperField { TF_X = 0, TF_Y, TF_R, TF_SIG, TF_NU, TF_DV, TF_COUNT };
struct TaperTable {
  double* base;
  int64_t stride;
  __host__ __device__ const double* f(int k) const { return base + (int64_t)k * stride; }
  __host__ __device__ double* fw(int k) const { return base + (int64_t)k * stride; }
};
void launch_taper_site_stage(int64_t n, int p, const double* dX, int64_t ldx, const double* dlocs, int64_t ldl,
                             const double* dtheta6, double lim0, double lim1, int mode, int pred_rows, TaperTable T,
                             cudaStream_t st);
enum TaperSinkKind { TS_VECTOR = 0, TS_LOWER = 1, TS_ROWS = 2, TS_TILED = 3 };
struct TaperSink {
  int kind;
  double* out;          // TS_VECTOR: nnz values in pattern order
  const double* taper;  // TS_LOWER / TS_ROWS / TS_TILED: taper values on the pattern, multiplied in
  const int* inv;       // caller index -> position in the context's ordering
  double* A;            // dense sink; TS_TILED: the tile pool
  int64_t ld;           // TS_TILED: number of tile columns T
  int64_t row0;         // TS_ROWS: first pattern row of the block; TS_TILED: number of stored tiles
  // TS_TILED: the tile map, int64 [T + 1 column starts][stored tiles: tile row][stored tiles: element offset of the
  // tile in the pool][T: leading dimension of column panel J]; the rows of a column are sorted, diagonal first
  const int64_t* tiles;
};
// the tiled sink runs in instantiations of taper_entries_kernel<mode + kTaperTiled> of their own
constexpr int kTaperTiled = 8;
// entries [e0, e0 + count) of the pattern (nrows rows)
void launch_taper_entries(int64_t e0, int64_t count, int64_t nrows, const int* dcol, const int* drow, TaperTable R,
                          TaperTable C, int square, int mode, double nu_fixed, TaperSink S, cudaStream_t st);
void launch_taper_pad_diag(int64_t n, int64_t n_pad, double* A, int64_t ld, cudaStream_t st);

// ---- chol.cu -------------------------------------------------------------
struct CholWorkspace {
  double* winv;               // (n_pad/kTile) inverted diagonal tiles, kTile x kTile each
  int* info;                  // device flag: 0 ok, k > 0 first non-positive pivot (1-based)
  cudaStream_t panel_stream;  // high-priority side stream for the look-ahead panel
  cudaEvent_t ev_a, ev_p;
  cudaEvent_t ev_k0, ev_k1;  // bracket the largest trailing-update launch (roofline measurement)
  // dataflow forward substitution (solve.cu, solve_workspace_create): control words, work-unit table, partial sums
  unsigned* solve_ctrl;   // [0] ticket, [1] front (rows of Y finished), [2] error, [4 + I] finished partial units of row I
  int* solve_units;       // 4 ints per unit: tile row I, first tile column J0, end J1, chunk index
  double* solve_part;     // (I * solve_nchunks + chunk) * kSolveMaxRhs * kTile doubles
  int solve_nunits, solve_nchunks;
  // split-int8 trailing update (syrk_i8.cu): int8 slices of the rows below one outer panel and their row scales;
  // null when the library was built without syrk_i8.cu or the workspace was created without it
  int8_t* i8_slices;
  double* i8_scale;
};
constexpr int kSolveMaxRhs = 8;   // right-hand sides per launch of the substitution kernels
constexpr int kSolveChunk = 16;   // tile columns per work unit (2 MB of L)
// with_i8: also the slice workspace of the split-int8 trailing update, when n_pad reaches it (kSyrkI8MinPad)
int chol_workspace_create(int64_t n_pad, CholWorkspace* ws, bool with_i8 = false);
void chol_workspace_destroy(CholWorkspace* ws);
// tiles [J0, J0+jb) of one outer panel (potrf + panel solve + in-panel update) on stream st; A is the
// address element (0,0) of the full matrix would have (only columns of the panel are touched)
void factor_panel(double* A, int64_t n_pad, int64_t ld, const CholWorkspace& ws, int64_t J0, int64_t jb,
                  cudaStream_t st);
int chol_factor(double* A, int64_t n_pad, int64_t ld, CholWorkspace ws, cudaStream_t st);
int chol_outer(int64_t n_pad);  // tiles per outer panel of chol_factor
// diagonal tile: Cholesky in place (leading dimension ld) and its explicit inverse into Winv (128 x 128); the first
// failing pivot sets *info = first_index + its 1-based order
void launch_potrf_tile(double* A, int64_t ld, double* Winv, int* info, int first_index, cudaStream_t st);
void launch_gemm_nt(int mode, int64_t M, int64_t N, int64_t K, const double* A, int64_t lda, const double* B,
                    int64_t ldb, double* C, int64_t ldc, int lower_only, cudaStream_t st);

// ---- syrk_i8.cu: the K = 768 trailing update C -= P P^T as exact products of int8 slices on the tensor cores
// (tcgen05, kind::i8), combined in FP64.  syrk_i8.cu fills g_syrk_i8 when it is linked in; a build of the sources
// without it (the host emulation of the tests) leaves the entries null and chol_factor keeps to the DMMA GEMM.
constexpr int kSyrkI8K = 768;                 // panel width the update is built for (chol_outer = 6 tiles)
constexpr int64_t kSyrkI8MinPad = 16384;      // n_pad from which chol_factor runs K = 768 panels
constexpr int64_t kSyrkI8BytesPerRow = 8 * kSyrkI8K;  // 8 int8 slices per row
struct SyrkI8Ops {
  // rows [0, m) of P (m x 768, column-major, m a multiple of 128) -> slices q and row scales
  void (*split)(const double* P, int64_t ld, int64_t m, int8_t* q, double* scale, cudaStream_t st);
  // C[M x N] -= P_a P_b^T over the lower 128 x 64 tiles (lower_only) or all of them, where P_a is rows
  // [a_row0, a_row0 + M) of the split panel and P_b rows [b_row0, b_row0 + N); a_row0, b_row0 multiples of 128.
  // A device wait that gave up (a bug) sets *info (device) to COCONS_ERR_CUDA if it was 0.
  void (*update)(int64_t M, int64_t N, const int8_t* q, const double* scale, int64_t a_row0, int64_t b_row0,
                 double* C, int64_t ldc, int lower_only, int* info, cudaStream_t st);
};
extern SyrkI8Ops g_syrk_i8;

// ---- solve.cu ------------------------------------------------------------
void launch_logdet(const double* L, int64_t n, int64_t ld, double* out, cudaStream_t st);
void forward_solve(const double* L, int64_t n_pad, int64_t ld, const double* winv, double* B, int64_t ldb, int nrhs,
                   cudaStream_t st);
int solve_workspace_create(int64_t n_pad, CholWorkspace* ws);
}  // namespace cocons
#include <vector>
namespace cocons {
int build_solve_units(int64_t T, std::vector<int>* out);  // host: work units of the dataflow substitution, issue order
void solve_workspace_destroy(CholWorkspace* ws);
// L Y = B with the dataflow kernel when ws carries a solve workspace (else the cooperative kernel above); a
// stalled dependency wait (which would be a bug) is reported through *info_dev = COCONS_ERR_CUDA instead of hanging
void forward_solve_ws(const double* L, int64_t n_pad, int64_t ld, const CholWorkspace& ws, double* B, int64_t ldb,
                      int nrhs, cudaStream_t st);
void launch_gram(const double* Y, int64_t n, int64_t ldy, int k, double* G, cudaStream_t st);

}  // namespace cocons

#endif
