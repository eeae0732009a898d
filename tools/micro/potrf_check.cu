// Standalone check + timing of the two diagonal-tile kernels (csrc/chol.cu): L L^T = A, W L = I against a
// host long-double factorisation, non-PD detection, and microseconds per launch over 200 independent tiles.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a tools/micro/potrf_check.cu -o tools/micro/potrf_check
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../../cocons_b200/csrc/chol.cu"
namespace cocons { void note_launch(int) {} void set_error(const char*, ...) {} }

static void host_chol(const std::vector<double>& A, std::vector<long double>& L, int n) {
  L.assign((size_t)n * n, 0.0L);
  for (int j = 0; j < n; ++j) {
    long double d = A[j * n + j];
    for (int k = 0; k < j; ++k) d -= L[k * n + j] * L[k * n + j];
    d = sqrtl(d);
    L[j * n + j] = d;
    for (int i = j + 1; i < n; ++i) {
      long double v = A[j * n + i];
      for (int k = 0; k < j; ++k) v -= L[k * n + i] * L[k * n + j];
      L[j * n + i] = v / d;
    }
  }
}

int main() {
  const int n = 128, reps = 200;
  double *dA, *dW;
  int* dinfo;
  cudaMalloc(&dA, sizeof(double) * n * n * reps);
  cudaMalloc(&dW, sizeof(double) * n * n * reps);
  cudaMalloc(&dinfo, 4);
  cudaFuncSetAttribute(cocons::potrf_tile_blocked_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       cocons::kPotrfBlockedSmem);
  for (int cas = 0; cas < 3; ++cas) {
    std::vector<double> A((size_t)n * n);
    srand(7 + cas);
    if (cas == 0) {
      for (int j = 0; j < n; ++j)
        for (int i = 0; i < n; ++i) A[j * n + i] = (i == j ? 4.0 : 0.0) + 1.0 / (1.0 + abs(i - j));
    } else {  // Gram matrix of random vectors + ridge: condition number ~1e3 (cas 1) / ~1e7 (cas 2)
      const int m = 160;
      std::vector<double> G((size_t)n * m);
      for (auto& g : G) g = rand() / (double)RAND_MAX - 0.5;
      const double ridge = cas == 1 ? 1e-1 : 1e-6;
      for (int j = 0; j < n; ++j)
        for (int i = 0; i < n; ++i) {
          double sacc = 0;
          for (int k = 0; k < m; ++k) sacc += G[i * m + k] * G[j * m + k] * (k < 100 || cas == 1 ? 1.0 : 1e-4);
          A[j * n + i] = sacc + (i == j ? ridge : 0.0);
        }
    }
    std::vector<long double> Lh;
    host_chol(A, Lh, n);
    for (int variant = 1; variant <= 2; ++variant) {
      cudaMemset(dinfo, 0, 4);
      cudaMemcpy(dA, A.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice);
      if (variant == 1)
        cocons::potrf_tile_kernel<<<1, 256>>>(dA, n, dW, dinfo, 0);
      else
        cocons::potrf_tile_blocked_kernel<0><<<1, 256, cocons::kPotrfBlockedSmem>>>(dA, n, dW, dinfo, 0);
      cudaError_t e = cudaDeviceSynchronize();
      std::vector<double> L((size_t)n * n), W((size_t)n * n);
      int info = -1;
      cudaMemcpy(L.data(), dA, sizeof(double) * n * n, cudaMemcpyDeviceToHost);
      cudaMemcpy(W.data(), dW, sizeof(double) * n * n, cudaMemcpyDeviceToHost);
      cudaMemcpy(&info, dinfo, 4, cudaMemcpyDeviceToHost);
      double errL = 0, errWL = 0, upper = 0, lmax = 0;
      for (int j = 0; j < n; ++j)
        for (int i = 0; i < n; ++i) {
          if (i < j) upper = fmax(upper, fmax(fabs(L[j * n + i]), fabs(W[j * n + i])));
          else {
            errL = fmax(errL, fabs((double)(L[j * n + i] - Lh[j * n + i])));
            lmax = fmax(lmax, fabs((double)Lh[j * n + i]));
          }
        }
      for (int j = 0; j < n; ++j)      // (W L)[i][j]
        for (int i = 0; i < n; ++i) {
          long double sacc = 0;
          for (int k = 0; k < n; ++k) sacc += (long double)W[k * n + i] * (long double)L[j * n + k];
          errWL = fmax(errWL, fabs((double)(sacc - (i == j ? 1.0L : 0.0L))));
        }
      printf("case %d variant %d: cuda=%s info=%d  max|L-Lref|=%.3e (|L|max %.2e)  max|W L - I|=%.3e  upper=%.1e\n", cas,
             variant, cudaGetErrorString(e), info, errL, lmax, errWL, upper);
    }
  }
  // non-PD: pivot 37 (1-based 38 + first_index 1000) becomes non-positive
  {
    std::vector<double> A((size_t)n * n, 0.0);
    for (int i = 0; i < n; ++i) A[i * n + i] = 2.0;
    A[37 * n + 37] = -1.0;
    for (int variant = 1; variant <= 2; ++variant) {
      cudaMemset(dinfo, 0, 4);
      cudaMemcpy(dA, A.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice);
      if (variant == 1)
        cocons::potrf_tile_kernel<<<1, 256>>>(dA, n, dW, dinfo, 1000);
      else
        cocons::potrf_tile_blocked_kernel<0><<<1, 256, cocons::kPotrfBlockedSmem>>>(dA, n, dW, dinfo, 1000);
      cudaDeviceSynchronize();
      int info = -1;
      cudaMemcpy(&info, dinfo, 4, cudaMemcpyDeviceToHost);
      printf("non-PD variant %d: info=%d (expected 1038)\n", variant, info);
    }
  }
  // timing: 200 independent tiles back to back
  {
    std::vector<double> A((size_t)n * n);
    for (int j = 0; j < n; ++j)
      for (int i = 0; i < n; ++i) A[j * n + i] = (i == j ? 4.0 : 0.0) + 1.0 / (1.0 + abs(i - j));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0), cudaEventCreate(&e1);
    for (int variant = 1; variant <= 2; ++variant) {
      for (int pass = 0; pass < 2; ++pass) {
        for (int r = 0; r < reps; ++r)
          cudaMemcpy(dA + (size_t)r * n * n, A.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice);
        cudaMemset(dinfo, 0, 4);
        cudaDeviceSynchronize();
        cudaEventRecord(e0);
        for (int r = 0; r < reps; ++r) {
          if (variant == 1)
            cocons::potrf_tile_kernel<<<1, 256>>>(dA + (size_t)r * n * n, n, dW + (size_t)r * n * n, dinfo, 0);
          else
            cocons::potrf_tile_blocked_kernel<0><<<1, 256, cocons::kPotrfBlockedSmem>>>(dA + (size_t)r * n * n, n,
                                                                                     dW + (size_t)r * n * n, dinfo, 0);
        }
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (pass == 1) printf("variant %d: %.2f us per tile (200 launches back to back)\n", variant, 1e3 * ms / reps);
      }
    }
  }
#ifdef COCONS_POTRF_PROBE
  {
    long long q[64];
    cudaMemcpyFromSymbol(q, cocons::g_probe_b, sizeof(q));
    printf("blocked kernel clocks (last launch): load %lld P1(0) %lld", q[1] - q[0], q[2] - q[1]);
    for (int s = 0; s < 8; ++s) printf(" | s=%d P2 %lld P3+P1 %lld", s, q[3 + 3 * s] - q[2 + 3 * s], q[4 + 3 * s] - q[3 + 3 * s]);
    printf(" | store %lld | total %lld\n", q[30] - q[25], q[30] - q[0]);
  }
#endif
  return 0;
}
