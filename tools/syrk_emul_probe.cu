// The lower-right quadrant update of a split Cholesky factorisation, A22 -= L21 L21' (L21: rows [128 hs, npad) x columns
// [0, 128 hs)): the rank-512 DMMA trailing updates it replaces (k_gemm, M_TRAIL_COL, one launch per panel of 4 block
// columns over the whole quadrant) against the INT8 modular emulation of dgp_lauum8.cuh (k_l8_convert + k_l8_gemm_ab in
// its full-K lower-tile mode + the accumulating k_l8_recon_ab, the launches of syrk_i8 in dgp_api.cu), timed with CUDA
// events, and sampled entries checked bit for bit against the exact product of the converted operands (host 128-bit
// integers), rounded once and subtracted from the old entry.
// Built and run by syrk_emul_probe.py.   usage: syrk_emul_probe npad:hs [npad:hs ...]   (one JSON line per case on stdout)
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

static __device__ double hgen(unsigned long long i, unsigned long long k, unsigned long long salt) {
  unsigned long long x = (i * 0x9E3779B97F4A7C15ull) ^ ((k + salt) * 0xBF58476D1CE4E5B9ull);
  x ^= x >> 31; x *= 0x94D049BB133111EBull; x ^= x >> 29;
  const double u = (double)(x >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0;
  return u * exp2(-(double)((x >> 3) & 7));   // several binades per row
}

// L lower triangular, A lower triangular with the diagonal blocks in full and garbage above them
__global__ void k_gen(double* L, double* A, int npad) {
  const int i = blockIdx.x;
  for (int k = threadIdx.x; k < npad; k += blockDim.x) {
    const size_t o = (size_t)i * npad + k;
    L[o] = k <= i ? hgen(i, k, 2) + (k == i ? 4.0 : 0.0) : 0.0;
    A[o] = k / 128 <= i / 128 ? hgen(i, k, 3) + (k == i ? 64.0 : 0.0) : 1e300;
  }
}

static CUtensorMap map_f64(PFN_encodeTiled e, double* p, int npad) {
  CUtensorMap m;
  cuuint64_t dims[2] = {(cuuint64_t)npad, (cuuint64_t)npad}, str[1] = {(cuuint64_t)npad * 8};
  cuuint32_t box[2] = {BK, 64}, es[2] = {1, 1};
  if (e(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, p, dims, str, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
    fprintf(stderr, "map f64\n"); exit(1);
  }
  return m;
}

static CUtensorMap map_i8(PFN_encodeTiled e, int8_t* p, long long rows, long long kw) {
  CUtensorMap m;
  cuuint64_t dims[3] = {(cuuint64_t)kw, (cuuint64_t)rows, (cuuint64_t)L8_NMOD}, str[2] = {(cuuint64_t)kw, (cuuint64_t)(kw * rows)};
  cuuint32_t box[3] = {128, 128, 1}, es[3] = {1, 1, 1};
  if (e(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, p, dims, str, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
    fprintf(stderr, "map i8\n"); exit(1);
  }
  return m;
}

int main(int argc, char** argv) {
  PFN_encodeTiled encode = enc();
  cudaFuncSetAttribute(k_gemm<INIT_LOAD, EPI_STORE>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL);
  cudaFuncSetAttribute(k_l8_gemm_ab, cudaFuncAttributeMaxDynamicSharedMemorySize, L8_SMEM);
  for (int a = 1; a < argc; a++) {
    int npad = 0, hs = 0;
    if (sscanf(argv[a], "%d:%d", &npad, &hs) != 2 || npad % 128 || hs % 4 || hs <= 0 || 128 * hs >= npad) {
      fprintf(stderr, "bad case %s\n", argv[a]); return 1;
    }
    const int nb = npad / 128, r = nb - hs;
    const size_t nn = (size_t)npad * npad;
    const long long kw = 128LL * hs, rows = 128LL * r;
    double *L, *A, *A0;
    int8_t* R;
    int* sexp;
    CKE(cudaMalloc(&L, nn * 8)); CKE(cudaMalloc(&A, nn * 8)); CKE(cudaMalloc(&A0, nn * 8));
    CKE(cudaMalloc(&R, (size_t)L8_NMOD * rows * (kw + rows))); CKE(cudaMalloc(&sexp, rows * 4));
    k_gen<<<npad, 256>>>(L, A0, npad);
    CKE(cudaGetLastError());
    const size_t o = (size_t)hs * 128;
    // DMMA: the rank-512 updates of the panels [0, hs) applied to the quadrant, one launch per panel
    CUtensorMap tmL = map_f64(encode, L, npad);
    BatchTab bt;
    memset(&bt, 0, sizeof(bt));
    dgp_spec spec;
    memset(&spec, 0, sizeof(spec));
    auto dmma = [&]() {
      for (int pb = 0; pb < hs; pb += 4) {
        GemmArgs g;
        memset(&g, 0, sizeof(g));
        g.mode = M_TRAIL_COL; g.step = pb; g.nb = nb; g.n = npad; g.ldc = npad;
        g.aux0 = hs | (r << 16); g.aux1 = 4; g.aux2 = 1; g.ntiles = r * 2 * r; g.C = A; g.sign = -1.0;
        k_gemm<INIT_LOAD, EPI_STORE><<<g.ntiles, GEMM_THREADS, SM_TOTAL>>>(tmL, tmL, spec, g, bt);
      }
    };
    int8_t* PA = R;
    int8_t* PC = PA + L8_NMOD * rows * kw;
    const CUtensorMap ta = map_i8(encode, PA, rows, kw);
    auto emul = [&](cudaEvent_t* ev) {
      cudaEventRecord(ev[0]);
      k_l8_convert<<<(unsigned)rows, 256>>>(L + o * npad, npad, (int)kw, l8_bits(kw), false, false, PA, kw, rows * kw, sexp);
      cudaEventRecord(ev[1]);
      k_l8_gemm_ab<<<L8_NMOD * l8_slots(r), 128, L8_SMEM>>>(ta, ta, r, r, hs, L8_KFULL_SYRK, PC);
      cudaEventRecord(ev[2]);
      k_l8_recon_ab<<<r * (r + 1) / 2, 256>>>(PC, r, r, sexp, sexp, -1.0, A + o * npad + o, npad, true);
      cudaEventRecord(ev[3]);
    };
    cudaEvent_t ev[6];
    for (auto& e : ev) cudaEventCreate(&e);
    CKE(cudaMemcpy(A, A0, nn * 8, cudaMemcpyDeviceToDevice));
    dmma(); emul(ev + 2);
    CKE(cudaGetLastError());
    CKE(cudaDeviceSynchronize());
    const int reps = 3;
    float t_d = 0, t_c = 0, t_g = 0, t_r = 0, x;
    for (int q = 0; q < reps; q++) {
      CKE(cudaMemcpy(A, A0, nn * 8, cudaMemcpyDeviceToDevice));
      cudaEventRecord(ev[0]); dmma(); cudaEventRecord(ev[1]);
      CKE(cudaEventSynchronize(ev[1]));
      cudaEventElapsedTime(&x, ev[0], ev[1]); t_d += x;
      CKE(cudaMemcpy(A, A0, nn * 8, cudaMemcpyDeviceToDevice));
      emul(ev + 2);
      CKE(cudaEventSynchronize(ev[5]));
      cudaEventElapsedTime(&x, ev[2], ev[3]); t_c += x;
      cudaEventElapsedTime(&x, ev[3], ev[4]); t_g += x;
      cudaEventElapsedTime(&x, ev[4], ev[5]); t_r += x;
    }
    CKE(cudaGetLastError());
    t_d /= reps; t_c /= reps; t_g /= reps; t_r /= reps;
    // the last emulated run (from A0): 512 sampled entries of the lower tiles, diagonal blocks in full, and the tile corners
    std::vector<std::pair<int, int>> at;
    for (int k = 0; at.size() < 512; k++) {
      int i = (int)((k * 2654435761ull + 17) % rows), c = (int)((k * 40503ull + 5 + k * k) % rows);
      if (k < 8) { i = k & 1 ? (int)rows - 1 : 0; c = k & 2 ? i : i / 128 * 128 + ((k & 4) ? 127 : 0); }
      if (c / 128 > i / 128) std::swap(i, c);
      at.push_back({i, c});
    }
    std::vector<int> hsx(rows);
    CKE(cudaMemcpy(hsx.data(), sexp, rows * 4, cudaMemcpyDeviceToHost));
    auto row_of = [&](long long i) {
      std::vector<double> u(kw);
      CKE(cudaMemcpy(u.data(), L + (o + i) * npad, kw * 8, cudaMemcpyDeviceToHost));
      return u;
    };
    long long checked = 0, bad = 0;
    double maxrel = 0.0;
    // keep the emulated result in A0, regenerate the original matrix in A for the old entries
    CKE(cudaMemcpy(A0, A, nn * 8, cudaMemcpyDeviceToDevice));
    k_gen<<<npad, 256>>>(L, A, npad);
    CKE(cudaDeviceSynchronize());
    for (auto [i, c] : at) {
      const std::vector<double> ar = row_of(i), bc = row_of(c);
      __int128 s = 0;
      for (long long k = 0; k < kw; k++)
        s += (__int128)(long long)rint(ldexp(ar[k], hsx[i])) * (long long)rint(ldexp(bc[k], hsx[c]));
      const bool neg = s < 0;
      const double prod = (neg ? -1.0 : 1.0) * l8_round((u128)(neg ? -s : s), -(hsx[i] + hsx[c]));
      double old, got;
      CKE(cudaMemcpy(&old, A + (o + i) * npad + o + c, 8, cudaMemcpyDeviceToHost));
      CKE(cudaMemcpy(&got, A0 + (o + i) * npad + o + c, 8, cudaMemcpyDeviceToHost));
      volatile double want = old - prod;
      checked++;
      if (memcmp((const void*)&want, &got, 8) != 0) {
        if (bad < 5) fprintf(stderr, "npad=%d hs=%d (%d,%d): emulated %.17g exact %.17g\n", npad, hs, i, c, got, (double)want);
        bad++;
      }
    }
    // the DMMA result on the same entries (from the regenerated A), for the size of the difference
    dmma();
    CKE(cudaDeviceSynchronize());
    for (auto [i, c] : at) {
      double d, e;
      CKE(cudaMemcpy(&d, A + (o + i) * npad + o + c, 8, cudaMemcpyDeviceToHost));
      CKE(cudaMemcpy(&e, A0 + (o + i) * npad + o + c, 8, cudaMemcpyDeviceToHost));
      if (e != 0.0) maxrel = std::max(maxrel, fabs(d - e) / fabs(e));
    }
    // INT8 operations: 2 per multiply-add, 16 moduli, the lower tiles at full K; FP64 flops of the DMMA updates
    const double tiles = (double)r * (r + 1) / 2;
    const double ops = 16.0 * 2.0 * tiles * 128.0 * 128.0 * (double)kw;
    const double flops = 2.0 * (double)r * 128.0 * ((double)r * 128.0 + 128.0) / 2.0 * (double)kw;
    printf("{\"npad\": %d, \"hs\": %d, \"dmma_ms\": %.3f, \"dmma_tflops\": %.1f, \"convert_ms\": %.3f, \"i8_gemm_ms\": %.3f, "
           "\"recon_ms\": %.3f, \"emulated_ms\": %.3f, \"i8_tops\": %.1f, \"checked\": %lld, \"mismatches\": %lld, "
           "\"dmma_max_rel_diff\": %.3e}\n",
           npad, hs, t_d, flops / (t_d * 1e-3) / 1e12, t_c, t_g, t_r, t_c + t_g + t_r, ops / (t_g * 1e-3) / 1e12, checked,
           bad, maxrel);
    fflush(stdout);
    for (auto& e : ev) cudaEventDestroy(e);
    cudaFree(L); cudaFree(A); cudaFree(A0); cudaFree(R); cudaFree(sexp);
  }
  return 0;
}
