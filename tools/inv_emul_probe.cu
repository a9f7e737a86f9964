// One merge of the recursive triangular inverse (block ranges hb | w2): M' = U11 L21' and U12 = -M' T22' on the FP64 DMMA
// tile engine (k_gemm, M_INV_M / M_INV_U) against the INT8 modular emulation of dgp_lauum8.cuh (conversion of both
// operands + k_l8_gemm_ab + k_l8_recon_ab, the launches of inv_merge_i8 in dgp_api.cu), timed with CUDA events, and the
// emulated entries checked bit for bit against the exact product of the converted operands (host 128-bit integers).
// Built and run by inv_emul_probe.py.   usage: inv_emul_probe hb:w2 [hb:w2 ...]   (one JSON line per merge on stdout)
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

// U upper triangular, L lower, T (lower triangle of the work matrix A) lower triangular; the upper triangle of A outside
// the diagonal blocks holds garbage, as the scratch of earlier merges leaves it
__global__ void k_gen(double* U, double* L, double* A, int npad) {
  const int i = blockIdx.x;
  for (int k = threadIdx.x; k < npad; k += blockDim.x) {
    const size_t o = (size_t)i * npad + k;
    U[o] = k >= i ? hgen(i, k, 1) + (k == i ? 4.0 : 0.0) : 0.0;
    L[o] = k <= i ? hgen(i, k, 2) + (k == i ? 4.0 : 0.0) : 0.0;
    A[o] = k <= i ? hgen(i, k, 3) + (k == i ? 4.0 : 0.0) : (k / 128 == i / 128 ? 0.0 : 1e300);
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

struct Prod { float conv, gemm, recon; };

int main(int argc, char** argv) {
  PFN_encodeTiled encode = enc();
  cudaFuncSetAttribute(k_gemm<INIT_ZERO, EPI_STORE>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL);
  cudaFuncSetAttribute(k_l8_gemm_ab, cudaFuncAttributeMaxDynamicSharedMemorySize, L8_SMEM);
  for (int a = 1; a < argc; a++) {
    int hb = 0, w2 = 0;
    if (sscanf(argv[a], "%d:%d", &hb, &w2) != 2 || w2 > hb || w2 < 1) { fprintf(stderr, "bad merge %s\n", argv[a]); return 1; }
    const int nb = hb + w2, npad = 128 * nb;
    const size_t nn = (size_t)npad * npad;
    const long long r1 = 128LL * hb, r2 = 128LL * w2;
    double *U, *L, *A, *Me, *Ue;
    int8_t* R;
    int* sexp;
    CKE(cudaMalloc(&U, nn * 8)); CKE(cudaMalloc(&L, nn * 8)); CKE(cudaMalloc(&A, nn * 8));
    CKE(cudaMalloc(&Me, (size_t)r1 * r2 * 8)); CKE(cudaMalloc(&Ue, (size_t)r1 * r2 * 8));
    CKE(cudaMalloc(&R, nn * L8_NMOD)); CKE(cudaMalloc(&sexp, npad * 4));
    k_gen<<<npad, 256>>>(U, L, A, npad);
    CKE(cudaGetLastError());
    // DMMA: both products of the merge (pair 0 of level hb), as trtri_advance launches them
    CUtensorMap tmU = map_f64(encode, U, npad), tmL = map_f64(encode, L, npad), tmA = map_f64(encode, A, npad);
    GemmArgs g;
    memset(&g, 0, sizeof(g));
    g.nb = nb; g.n = npad; g.ldc = npad; g.aux0 = hb; g.aux1 = 1; g.ntiles = hb * 2 * hb;
    BatchTab bt;
    memset(&bt, 0, sizeof(bt));
    dgp_spec spec;
    memset(&spec, 0, sizeof(spec));
    auto dmma = [&]() {
      GemmArgs gm = g; gm.mode = M_INV_M; gm.C = A; gm.sign = 1.0;
      k_gemm<INIT_ZERO, EPI_STORE><<<gm.ntiles, GEMM_THREADS, SM_TOTAL>>>(tmU, tmL, spec, gm, bt);
      GemmArgs gu = g; gu.mode = M_INV_U; gu.C = U; gu.sign = -1.0;
      k_gemm<INIT_ZERO, EPI_STORE><<<gu.ntiles, GEMM_THREADS, SM_TOTAL>>>(tmA, tmA, spec, gu, bt);
    };
    // emulated: the launches of gemm_ab_i8 (dgp_api.cu) for M' -> Me and U12 -> Ue
    const double* T22 = A + (size_t)r1 * npad + r1;
    auto prod = [&](bool first, cudaEvent_t* ev) {
      const int kb = first ? hb : w2;
      const long long kw = 128LL * kb;
      int8_t* PA = R;
      int8_t* PB = PA + L8_NMOD * r1 * kw;
      int8_t* PC = PB + L8_NMOD * r2 * kw;
      const int b = l8_bits(kw);
      const CUtensorMap ta = map_i8(encode, PA, r1, kw), tb = map_i8(encode, PB, r2, kw);
      cudaEventRecord(ev[0]);
      if (first) {
        k_l8_convert<<<(unsigned)r1, 256>>>(U, npad, (int)kw, b, true, false, PA, kw, r1 * kw, sexp);
        k_l8_convert<<<(unsigned)r2, 256>>>(L + (size_t)r1 * npad, npad, (int)kw, b, false, false, PB, kw, r2 * kw, sexp + r1);
      } else {
        k_l8_convert<<<(unsigned)r1, 256>>>(Me, r2, (int)kw, b, false, false, PA, kw, r1 * kw, sexp);
        k_l8_convert<<<(unsigned)r2, 256>>>(T22, npad, (int)kw, b, false, true, PB, kw, r2 * kw, sexp + r1);
      }
      cudaEventRecord(ev[1]);
      k_l8_gemm_ab<<<L8_NMOD * 64 * ((hb + 7) / 8) * ((w2 + 7) / 8), 128, L8_SMEM>>>(ta, tb, hb, w2, kb, first, PC);
      cudaEventRecord(ev[2]);
      k_l8_recon_ab<<<hb * w2, 256>>>(PC, hb, w2, sexp, sexp + r1, first ? 1.0 : -1.0, first ? Me : Ue, r2);
      cudaEventRecord(ev[3]);
    };
    cudaEvent_t ev[6];
    for (auto& e : ev) cudaEventCreate(&e);
    dmma(); prod(true, ev + 2); prod(false, ev + 2);
    CKE(cudaGetLastError());
    CKE(cudaDeviceSynchronize());
    const int reps = hb >= 64 ? 3 : 10;
    float t_d = 0;
    Prod p1 = {0, 0, 0}, p2 = {0, 0, 0};
    for (int r = 0; r < reps; r++) {
      float x;
      cudaEventRecord(ev[0]); dmma(); cudaEventRecord(ev[1]);
      CKE(cudaEventSynchronize(ev[1]));
      cudaEventElapsedTime(&x, ev[0], ev[1]); t_d += x;
      for (int q = 0; q < 2; q++) {
        Prod& p = q ? p2 : p1;
        prod(q == 0, ev + 2);
        CKE(cudaEventSynchronize(ev[5]));
        cudaEventElapsedTime(&x, ev[2], ev[3]); p.conv += x;
        cudaEventElapsedTime(&x, ev[3], ev[4]); p.gemm += x;
        cudaEventElapsedTime(&x, ev[4], ev[5]); p.recon += x;
      }
    }
    CKE(cudaGetLastError());
    t_d /= reps;
    for (Prod* p : {&p1, &p2}) { p->conv /= reps; p->gemm /= reps; p->recon /= reps; }
    // exactness on sampled entries of both products (operands converted on the host from the device's row scales)
    std::vector<int> rows = {0, 1, 127, 128, (int)r1 / 2, (int)r1 - 129, (int)r1 - 128, (int)r1 - 1};
    std::vector<int> cols = {0, 1, 63, 64, 127, 128, (int)r2 / 2, (int)r2 - 65, (int)r2 - 64, (int)r2 - 1};
    for (int k = 0; k < 8; k++) {
      rows.push_back((int)((k * 2654435761ull + 17) % r1));
      cols.push_back((int)((k * 40503ull + 5) % r2));
    }
    for (auto* v : {&rows, &cols}) { std::sort(v->begin(), v->end()); v->erase(std::unique(v->begin(), v->end()), v->end()); }
    long long checked = 0, bad = 0;
    double maxrel = 0.0;
    for (int q = 0; q < 2; q++) {
      const bool first = q == 0;
      const long long kw = first ? r1 : r2;
      prod(first, ev + 2);
      CKE(cudaDeviceSynchronize());
      std::vector<int> hs(r1 + r2);
      CKE(cudaMemcpy(hs.data(), sexp, (r1 + r2) * 4, cudaMemcpyDeviceToHost));
      auto row_of = [&](const double* base, long long ld, long long r, long long lo, long long hi) {
        std::vector<double> u(kw);
        CKE(cudaMemcpy(u.data(), base + r * ld, kw * 8, cudaMemcpyDeviceToHost));
        for (long long k = 0; k < kw; k++) if (k < lo || k >= hi) u[k] = 0.0;
        return u;
      };
      for (int r : rows) {
        const std::vector<double> ar = first ? row_of(U, npad, r, r / 128 * 128, kw) : row_of(Me, r2, r, 0, kw);
        std::vector<double> got(r2), ref(r2);
        CKE(cudaMemcpy(got.data(), (first ? Me : Ue) + (size_t)r * r2, r2 * 8, cudaMemcpyDeviceToHost));
        CKE(cudaMemcpy(ref.data(), (first ? A : U) + (size_t)r * npad + r1, r2 * 8, cudaMemcpyDeviceToHost));
        for (int c : cols) {
          const std::vector<double> bc = first ? row_of(L + (size_t)r1 * npad, npad, c, 0, kw)
                                               : row_of(T22, npad, c, 0, c / 64 * 64 + 64);
          __int128 s = 0;
          for (long long k = 0; k < kw; k++)
            s += (__int128)(long long)rint(ldexp(ar[k], hs[r])) * (long long)rint(ldexp(bc[k], hs[r1 + c]));
          const bool neg = s < 0;
          double want = (neg ? -1.0 : 1.0) * l8_round((u128)(neg ? -s : s), -(hs[r] + hs[r1 + c]));
          if (!first) want = -want;
          checked++;
          if (memcmp(&want, &got[c], 8) != 0) {
            if (bad < 5) fprintf(stderr, "hb=%d w2=%d %s (%d,%d): emulated %.17g exact %.17g\n", hb, w2, first ? "M'" : "U12", r, c, got[c], want);
            bad++;
          }
          if (first && want != 0.0) maxrel = std::max(maxrel, fabs(ref[c] - want) / fabs(want));
        }
      }
    }
    // INT8 operations of both products: 2 per multiply-add, 16 moduli, the k blocks each tile runs
    double ops = 0.0;
    for (int i = 0; i < hb; i++) ops += (double)(hb - i) * w2;
    for (int c = 0; c < w2; c++) ops += (double)(c + 1) * hb;
    ops *= 16.0 * 2.0 * 128.0 * 128.0 * 128.0;
    const double emul = p1.conv + p1.gemm + p1.recon + p2.conv + p2.gemm + p2.recon;
    printf("{\"hb\": %d, \"w2\": %d, \"dmma_ms\": %.3f, \"m_convert_ms\": %.3f, \"m_i8_gemm_ms\": %.3f, \"m_recon_ms\": %.3f, "
           "\"u_convert_ms\": %.3f, \"u_i8_gemm_ms\": %.3f, \"u_recon_ms\": %.3f, \"emulated_ms\": %.3f, \"i8_tops\": %.1f, "
           "\"checked\": %lld, \"mismatches\": %lld, \"dmma_max_rel_diff_m\": %.3e}\n",
           hb, w2, t_d, p1.conv, p1.gemm, p1.recon, p2.conv, p2.gemm, p2.recon, emul,
           ops / ((p1.gemm + p2.gemm) * 1e-3) / 1e12, checked, bad, maxrel);
    fflush(stdout);
    for (auto& e : ev) cudaEventDestroy(e);
    cudaFree(U); cudaFree(L); cudaFree(A); cudaFree(Me); cudaFree(Ue); cudaFree(R); cudaFree(sexp);
  }
  return 0;
}
