// LAUUM K^-1 = U U' (lower tiles): the FP64 DMMA tile engine (k_gemm, M_LAUUM) against the INT8 modular emulation
// (dgp_lauum8.cuh: conversion + tcgen05 GEMM + CRT reconstruction), timed with CUDA events, and the emulated entries
// checked bit for bit against the exact product of the converted operands (host 128-bit integers) on sampled entries.
// Built and run by lauum_emul_probe.py.   usage: lauum_emul_probe n1 [n2 ...]   (one JSON line per size on stdout)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <vector>
#include <algorithm>
#include "../include/dgp.h"
#include "../discontinuum_b200/csrc/dgp_lauum8.cuh"

using namespace dgp;

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

#define CKE(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s: %s (line %d)\n", #x, cudaGetErrorString(e_), __LINE__); exit(1); } } while (0)

static PFN_encodeTiled enc() {
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
    fprintf(stderr, "no cuTensorMapEncodeTiled\n"); exit(1);
  }
  return (PFN_encodeTiled)p;
}

static __device__ double ugen(unsigned long long i, unsigned long long k) {
  unsigned long long x = i * 0x9E3779B97F4A7C15ull ^ (k + 0x632BE59BD9B4E019ull) * 0xBF58476D1CE4E5B9ull;
  x ^= x >> 31; x *= 0x94D049BB133111EBull; x ^= x >> 29;
  const double u = (double)(x >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0;   // [-1, 1)
  // an inverse Cholesky factor's rows decay away from the diagonal and span several binades
  return (k == i ? 4.0 : u) * exp2(-(double)((x >> 3) & 7)) / (1.0 + 0.01 * (double)(k - i));
}

__global__ void k_gen_u(double* U, int npad) {
  const int i = blockIdx.x;
  for (int k = threadIdx.x; k < npad; k += blockDim.x) U[(size_t)i * npad + k] = k >= i ? ugen(i, k) : 0.0;
}

int main(int argc, char** argv) {
  PFN_encodeTiled encode = enc();
  cudaFuncSetAttribute(k_gemm<INIT_ZERO, EPI_STORE>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL);
  cudaFuncSetAttribute(k_l8_gemm, cudaFuncAttributeMaxDynamicSharedMemorySize, L8_SMEM);
  for (int a = 1; a < argc; a++) {
    const int n = atoi(argv[a]), npad = (n + 127) / 128 * 128, nb = npad / 128;
    const size_t nn = (size_t)npad * npad;
    double *U, *Kd, *Ke;
    int8_t *R, *D;
    int* sexp;
    CKE(cudaMalloc(&U, nn * 8)); CKE(cudaMalloc(&Kd, nn * 8)); CKE(cudaMalloc(&Ke, nn * 8));
    CKE(cudaMalloc(&R, nn * L8_NMOD)); CKE(cudaMalloc(&D, (size_t)npad * 128 * L8_NMOD)); CKE(cudaMalloc(&sexp, npad * 4));
    CKE(cudaMemset(Kd, 0, nn * 8)); CKE(cudaMemset(Ke, 0, nn * 8));
    k_gen_u<<<npad, 256>>>(U, npad);
    CKE(cudaGetLastError());
    // DMMA LAUUM
    CUtensorMap tmU, tmR;
    {
      cuuint64_t dims[2] = {(cuuint64_t)npad, (cuuint64_t)npad}, str[1] = {(cuuint64_t)npad * 8};
      cuuint32_t box[2] = {BK, 64}, es[2] = {1, 1};
      if (encode(&tmU, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, U, dims, str, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                 CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) { fprintf(stderr, "map U\n"); return 1; }
      cuuint64_t d3[3] = {(cuuint64_t)npad, (cuuint64_t)npad, (cuuint64_t)L8_NMOD}, s3[2] = {(cuuint64_t)npad, (cuuint64_t)nn};
      cuuint32_t b3[3] = {128, 128, 1}, e3[3] = {1, 1, 1};
      if (encode(&tmR, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, R, d3, s3, b3, e3, CU_TENSOR_MAP_INTERLEAVE_NONE,
                 CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) { fprintf(stderr, "map R\n"); return 1; }
    }
    GemmArgs g;
    memset(&g, 0, sizeof(g));
    g.mode = M_LAUUM; g.nb = nb; g.n = n; g.C = Kd; g.ldc = npad; g.sign = 1.0; g.ntiles = lauum_slots(nb);
    BatchTab bt;
    memset(&bt, 0, sizeof(bt));
    dgp_spec spec;
    memset(&spec, 0, sizeof(spec));
    const int b = l8_bits(npad);
    auto dmma = [&]() { k_gemm<INIT_ZERO, EPI_STORE><<<g.ntiles, GEMM_THREADS, SM_TOTAL>>>(tmU, tmU, spec, g, bt); };
    auto conv = [&]() { k_l8_convert<<<npad, 256>>>(U, npad, npad, b, true, false, R, npad, (long long)nn, sexp); };
    auto gemm = [&]() { k_l8_gemm<<<L8_NMOD * l8_slots(nb), 128, L8_SMEM>>>(tmR, nb, R, D, npad); };
    auto recon = [&]() { k_l8_recon<<<nb * (nb + 1) / 2, 256>>>(R, D, npad, sexp, Ke, npad); };
    dmma(); conv(); gemm(); recon();
    CKE(cudaGetLastError());
    CKE(cudaDeviceSynchronize());
    const int reps = npad >= 16384 ? 3 : 10;
    cudaEvent_t ev[5];
    for (auto& e : ev) cudaEventCreate(&e);
    float t_d = 0, t_c = 0, t_g = 0, t_r = 0;
    for (int r = 0; r < reps; r++) {
      cudaEventRecord(ev[0]); dmma(); cudaEventRecord(ev[1]); conv(); cudaEventRecord(ev[2]); gemm(); cudaEventRecord(ev[3]);
      recon(); cudaEventRecord(ev[4]);
      CKE(cudaEventSynchronize(ev[4]));
      float x;
      cudaEventElapsedTime(&x, ev[0], ev[1]); t_d += x;
      cudaEventElapsedTime(&x, ev[1], ev[2]); t_c += x;
      cudaEventElapsedTime(&x, ev[2], ev[3]); t_g += x;
      cudaEventElapsedTime(&x, ev[3], ev[4]); t_r += x;
    }
    CKE(cudaGetLastError());
    t_d /= reps; t_c /= reps; t_g /= reps; t_r /= reps;
    // exactness on sampled entries: rows of the first / last row blocks, diagonal blocks, the last row
    std::vector<int> rows = {0, 1, 127, 128, npad / 2, npad / 2 + 77, npad - 129, npad - 128, npad - 2, npad - 1};
    for (int k = 0; k < 22; k++) rows.push_back((int)((k * 2654435761ull + 17) % npad));
    std::sort(rows.begin(), rows.end());
    rows.erase(std::unique(rows.begin(), rows.end()), rows.end());
    std::vector<int> hs(npad);
    CKE(cudaMemcpy(hs.data(), sexp, npad * 4, cudaMemcpyDeviceToHost));
    auto conv_row = [&](int r) {   // the row as the device holds it, converted in host arithmetic
      std::vector<double> u(npad);
      CKE(cudaMemcpy(u.data(), U + (size_t)r * npad, npad * 8, cudaMemcpyDeviceToHost));
      std::vector<long long> v(npad);
      for (int k = 0; k < npad; k++) v[k] = (long long)rint(ldexp(u[k], hs[r]));
      return v;
    };
    long long checked = 0, bad = 0;
    double maxrel = 0.0;
    std::vector<std::vector<long long>> cache(rows.size());
    for (size_t a_ = 0; a_ < rows.size(); a_++) cache[a_] = conv_row(rows[a_]);
    for (size_t ia = 0; ia < rows.size(); ia++) {
      const int r = rows[ia];
      // columns: every sampled row in the lower block triangle, plus 64 columns of r's diagonal block
      std::vector<std::pair<int, const std::vector<long long>*>> cs;
      for (size_t ib = 0; ib < rows.size(); ib++) if (rows[ib] / 128 <= r / 128) cs.push_back({rows[ib], &cache[ib]});
      std::vector<std::vector<long long>> extra;
      for (int q = 0; q < 64; q++) extra.push_back(conv_row((r / 128) * 128 + 2 * q + (r & 1)));
      for (int q = 0; q < 64; q++) cs.push_back({(r / 128) * 128 + 2 * q + (r & 1), &extra[q]});
      std::vector<double> ke(npad), kd(npad);
      CKE(cudaMemcpy(ke.data(), Ke + (size_t)r * npad, npad * 8, cudaMemcpyDeviceToHost));
      CKE(cudaMemcpy(kd.data(), Kd + (size_t)r * npad, npad * 8, cudaMemcpyDeviceToHost));
      for (auto& pc : cs) {
        const int c = pc.first;
        const std::vector<long long>& vr = cache[ia];
        const std::vector<long long>& vc = *pc.second;
        __int128 s = 0;
        for (int k = std::max(r, c) / 128 * 128; k < npad; k++) s += (__int128)vr[k] * vc[k];
        const bool neg = s < 0;
        const double want = (neg ? -1.0 : 1.0) * l8_round((u128)(neg ? -s : s), -(hs[r] + hs[c]));
        checked++;
        if (memcmp(&want, &ke[c], 8) != 0) {
          if (bad < 5) fprintf(stderr, "n=%d (%d,%d): emulated %.17g exact %.17g dmma %.17g\n", n, r, c, ke[c], want, kd[c]);
          bad++;
        }
        if (want != 0.0) maxrel = std::max(maxrel, fabs(kd[c] - want) / fabs(want));
      }
    }
    const double ops = 16.0 * (double)npad * npad * npad / 3.0;
    printf("{\"n\": %d, \"b\": %d, \"dmma_lauum_ms\": %.3f, \"convert_ms\": %.3f, \"i8_gemm_ms\": %.3f, \"recon_ms\": %.3f, "
           "\"emulated_ms\": %.3f, \"i8_tops\": %.1f, \"checked\": %lld, \"mismatches\": %lld, \"dmma_max_rel_diff\": %.3e}\n",
           n, b, t_d, t_c, t_g, t_r, t_c + t_g + t_r, ops / (t_g * 1e-3) / 1e12, checked, bad, maxrel);
    fflush(stdout);
    for (auto& e : ev) cudaEventDestroy(e);
    cudaFree(U); cudaFree(Kd); cudaFree(Ke); cudaFree(R); cudaFree(D); cudaFree(sexp);
  }
  return 0;
}
