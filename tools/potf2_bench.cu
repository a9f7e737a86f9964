// Micro-benchmark / self-check of the diagonal-block kernel (development aid): k_potf2_v2 on one random SPD 128x128
// block: event timing of 200 back-to-back launches, the residuals max |L L' - A| and max |T L - I| (T = L^-1) and the
// agreement of U with T' (and, with P2_FULL set, of the contiguous copy DI with T), and, with -DP2_TIMING, the clock64
// stamps of its phases.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -DP2_TIMING -o tools/potf2_bench tools/potf2_bench.cu
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <vector>
#include <cuda.h>
#include <cuda_runtime.h>
#include "../include/dgp.h"
#include "../discontinuum_b200/csrc/dgp_cov.cuh"
#include "../discontinuum_b200/csrc/dgp_gemm.cuh"
#include "../discontinuum_b200/csrc/dgp_panel.cuh"
#include "../discontinuum_b200/csrc/dgp_potf2.cuh"
using namespace dgp;

int main() {
  const int ld = 256;
  const bool full = getenv("P2_FULL") != nullptr;
  std::vector<double> A(128 * ld, 0.0), G(128 * 128);
  srand(1);
  for (auto& g : G) g = rand() / (double)RAND_MAX - 0.5;
  for (int i = 0; i < 128; i++)
    for (int j = 0; j <= i; j++) {
      double s = (i == j) ? 1.0 : 0.0;
      for (int k = 0; k < 128; k++) s += G[i * 128 + k] * G[j * 128 + k] / 16.0;
      A[i * ld + j] = s;
      A[j * ld + i] = 777.0;  // garbage above the diagonal must be ignored
      if (i == j) A[i * ld + j] = s;
    }
  double *dA, *dL, *dU, *dDI, *dT, *scal;
  cudaMalloc(&dA, 128 * ld * 8); cudaMalloc(&scal, 64 * 8);
  cudaMalloc(&dL, 128 * ld * 8); cudaMalloc(&dU, 128 * ld * 8); cudaMalloc(&dDI, 128 * 128 * 8); cudaMalloc(&dT, 128 * ld * 8);
  cudaMemset(dL, 0xff, 128 * ld * 8); cudaMemset(dU, 0xff, 128 * ld * 8); cudaMemset(dT, 0xff, 128 * ld * 8);
  cudaMemcpy(dA, A.data(), 128 * ld * 8, cudaMemcpyHostToDevice);
  cudaMemset(scal, 0, 64 * 8);
  cudaFuncSetAttribute(k_potf2_v2, cudaFuncAttributeMaxDynamicSharedMemorySize, P2_SMEM);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int rep = 0; rep < 2; rep++) {
    const int iters = rep ? 200 : 3;
    cudaEventRecord(e0);
    for (int it = 0; it < iters; it++)
      k_potf2_v2<<<1, P2_THREADS, P2_SMEM>>>(dA, dL, dU, ld, full ? dDI : nullptr, scal, 0, dT, 1, P2Batch{});
    cudaEventRecord(e1); cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    if (rep) printf("k_potf2_v2: %.2f us per launch (%s)\n", ms * 1e3 / iters, cudaGetErrorString(cudaGetLastError()));
  }
  std::vector<double> L(128 * ld), U(128 * ld), DI(128 * 128), T(128 * ld);
  cudaMemcpy(L.data(), dL, 128 * ld * 8, cudaMemcpyDeviceToHost);
  cudaMemcpy(U.data(), dU, 128 * ld * 8, cudaMemcpyDeviceToHost);
  cudaMemcpy(DI.data(), dDI, 128 * 128 * 8, cudaMemcpyDeviceToHost);
  cudaMemcpy(T.data(), dT, 128 * ld * 8, cudaMemcpyDeviceToHost);
  double ra = 0, rt = 0, du = 0, dd = 0;
  for (int i = 0; i < 128; i++)
    for (int j = 0; j < 128; j++) {
      double llt = 0, tl = 0;
      for (int k = 0; k < 128; k++) { llt += L[i * ld + k] * L[j * ld + k]; tl += T[i * ld + k] * L[k * ld + j]; }
      if (j <= i) ra = fmax(ra, fabs(llt - A[i * ld + j]));
      rt = fmax(rt, fabs(tl - (i == j ? 1.0 : 0.0)));
      du = fmax(du, fabs(U[i * ld + j] - T[j * ld + i]));
      if (full) dd = fmax(dd, fabs(DI[i * 128 + j] - T[i * ld + j]));
    }
  printf("max |L L' - A| %.3e  |T L - I| %.3e  |U - T'| %.3e  |DI - T| %.3e\n", ra, rt, du, dd);
#ifdef P2_TIMING
  long long ts[64];
  cudaMemcpyFromSymbol(ts, p2_ts, sizeof(ts));
  printf("stamps (cycles from start): load %lld\n", ts[1] - ts[0]);
  for (int k = 0; k < 4; k++)
    printf(" k=%d pivots %lld  A-end %lld  (sync %lld)  B %lld  C %lld  D %lld\n", k, ts[2 + 6 * k] - (k ? ts[7 + 6 * (k - 1)] : ts[1]),
           ts[3 + 6 * k] - ts[2 + 6 * k], ts[4 + 6 * k] - ts[3 + 6 * k], ts[5 + 6 * k] - ts[4 + 6 * k], ts[6 + 6 * k] - ts[5 + 6 * k],
           ts[7 + 6 * k] - ts[6 + 6 * k]);
  printf(" inv row 3 %lld  outputs %lld  total %lld\n", ts[26] - ts[25], ts[27] - ts[26], ts[27] - ts[0]);
  long long wts[64];
  cudaMemcpyFromSymbol(wts, p2_wts, sizeof(wts));
  for (int b = 0; b < 2; b++)
    for (int k = 0; k < 4; k++) {
      printf(" barrier %d k=%d arrival of warps 0..7 (cycles after phase A start):", b, k);
      for (int w = 0; w < 8; w++) printf(" %lld", wts[b * 32 + k * 8 + w] - (k ? ts[7 + 6 * (k - 1)] : ts[1]));
      printf("\n");
    }
#endif
  return 0;
}
