// Ky^-1 = U U' (lower 128 x 128 tiles) on the INT8 tensor cores, exact to one rounding per entry (Ozaki scheme II).
//
//   1. k_l8_convert: row i of U is scaled by 2^s_i (s_i = b - 1 - e_i, |U_ik| < 2^e_i for the row's largest entry) and
//      rounded to an integer A'_ik, |A'| <= 2^(b-1); its residues modulo 16 pairwise-coprime odd moduli m_j < 256 are stored
//      as int8 in [-127, 127], one plane per modulus (the upper block triangle of the plane, diagonal blocks included).
//   2. k_l8_gemm: C_j = A_j A_j' mod m_j for every lower tile and modulus, tcgen05.mma kind::i8 with INT32 accumulators in
//      tensor memory (|C_j| <= npad 127^2 < 2^31, no overflow below L8_MAX_NPAD), operands by TMA through an mbarrier ring.
//      The int8 residues of the product go to the strictly lower block triangle of the same plane, those of the diagonal
//      tiles to a [plane][npad][128] side buffer (the operand still occupies the diagonal blocks).
//   3. k_l8_recon: the Chinese remainder theorem in 128-bit integer arithmetic gives C' = A' A'' exactly (|C'| < M / 2,
//      M = prod m_j ~ 2^124.95, which is what fixes b), rounded once to double and scaled by 2^-(s_r + s_c).
//
// The same kernels form C = sign A B' for the merges of the inverse (k_l8_gemm_ab, k_l8_recon_ab) and the quadrant update
// A22 -= L21 L21' of the split factorisation (L8_KFULL_SYRK, accumulating reconstruction); see dgp_api.cu.
//
// The result is a deterministic function of U and npad alone (no tiling or launch order enters it), so a batched
// launch reproduces a single-site one bit for bit.  b = l8_bits(npad) is the largest b with 2 npad 2^(2b-2) < M: 55 at
// npad = 16384 and 32768, one rounding of each operand at 2^-54 relative to its row's largest entry.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include "dgp_gemm.cuh"

namespace dgp {

constexpr int L8_NMOD = 16;
constexpr int L8_MAX_NPAD = 133120;   // npad * 127^2 < 2^31: the INT32 accumulators cannot overflow
constexpr int L8_STAGES = 3;
constexpr int L8_TILE_BYTES = 128 * 128;                  // one 128-row x 128-byte operand box
constexpr int L8_STAGE_BYTES = 2 * L8_TILE_BYTES;
constexpr int L8_SMEM = L8_STAGES * L8_STAGE_BYTES + 256 + 1024;   // ring + barriers + alignment slack

// modulus j, (M / m_j)^-1 mod m_j and M / m_j (two 64-bit halves)
struct L8Mod { int m, inv; unsigned long long hi, lo; };
__host__ __device__ constexpr L8Mod l8_mod(int j) {
  switch (j) {
    case 0: return {255, 124, 0x001f18e05cbc1ae2ull, 0x1840628c1d0eab21ull};
    case 1: return {253, 215, 0x001f57cee91aaed3ull, 0xb13bd5aa90a3870bull};
    case 2: return {251, 217, 0x001f97be33604007ull, 0x5aeecc265084316dull};
    case 3: return {247, 18, 0x00201ab7f3f2e8f7ull, 0xed81b166285ce059ull};
    case 4: return {241, 119, 0x0020e7557ecd67ddull, 0x2bb7e8cd9d26e3cfull};
    case 5: return {239, 134, 0x00212dd276392a9bull, 0x8a57f9bf447dfa11ull};
    case 6: return {233, 223, 0x0022088c11fd1c52ull, 0xa2c81cbeb3074387ull};
    case 7: return {229, 51, 0x0022a0bb3baa55d4ull, 0xa363a4836d7de373ull};
    case 8: return {227, 120, 0x0022eed5b17a3702ull, 0x7e7c340f4c9fb3d5ull};
    case 9: return {223, 174, 0x00238f3e8c7b4254ull, 0x0ba8e8142a692b01ull};
    case 10: return {217, 5, 0x00248af26a9d5709ull, 0xaff6b83a7971f977ull};
    case 11: return {211, 6, 0x002594f6e21ec7ebull, 0xa18e1d50c344af45ull};
    case 12: return {199, 152, 0x0027d91f7fd60625ull, 0x94243117e256fa29ull};
    case 13: return {197, 117, 0x002840b01013f936ull, 0xda84b8bd2982be53ull};
    case 14: return {193, 13, 0x00291641a3a4f7bfull, 0x49294bd2537d7e9full};
    default: return {191, 135, 0x002984652cbaccc5ull, 0x4f49e5694da9b2e1ull};
  }
}
constexpr unsigned long long L8_M_HI = 0x1ef9c77c5f5ec736ull, L8_M_LO = 0x28222990f19c75dfull;   // M = prod m_j

typedef unsigned __int128 u128;

// largest b with 2 npad 2^(2b-2) < M (depends on npad only)
constexpr int l8_bits(long long npad) {
  const u128 M = ((u128)L8_M_HI << 64) | L8_M_LO;
  int b = 2;
  while ((((u128)(2 * npad)) << (2 * (b + 1) - 2)) < M) ++b;
  return b;
}

// symmetric residue of a' = sign * a modulo m: a = a2 2^36 + a1 2^18 + a0, with a < 2^59 so that the 32-bit sum cannot
// overflow (a2 < 2^23); |A'| <= 2^(b-1) <= 2^58 at every npad >= 128
// (j a compile-time constant after unrolling: the divisions become multiplications)
static_assert(l8_bits(128) - 1 <= 58, "operands of the smallest size exceed the bound of l8_residue");
__host__ __device__ __forceinline__ int l8_residue(unsigned long long a, bool neg, int j) {
  const int m = l8_mod(j).m;
  const unsigned c18 = (1u << 18) % m, c36 = (unsigned)((1ull << 36) % m);
  const unsigned s = (unsigned)(a >> 36) * c36 + (unsigned)((a >> 18) & 0x3ffff) * c18 + (unsigned)(a & 0x3ffff);
  int r = (int)(s % m);
  if (neg) r = r ? m - r : 0;
  return r > m / 2 ? r - m : r;
}

// x 2^k, as ldexp: one multiplication by 2^k while that is a normal double (the exact product, rounded once if it is
// subnormal), instead of ldexp's general range handling on every call
__host__ __device__ __forceinline__ double l8_ldexp(double x, int k) {
  if (k < -1022 || k > 1023) return ldexp(x, k);
  const unsigned long long p = (unsigned long long)(k + 1023) << 52;
#ifdef __CUDA_ARCH__
  return x * __longlong_as_double((long long)p);
#else
  double f;
  memcpy(&f, &p, sizeof(f));
  return x * f;
#endif
}

// the 126-bit magnitude x, rounded once to double (round to nearest even), times 2^sc
__host__ __device__ __forceinline__ double l8_round(u128 x, int sc) {
  const unsigned long long hi = (unsigned long long)(x >> 64), lo = (unsigned long long)x;
  if (hi == 0) return l8_ldexp((double)lo, sc);
#ifdef __CUDA_ARCH__
  const int lz = __clzll((long long)hi);
#else
  const int lz = __builtin_clzll(hi);
#endif
  const int sh = 64 - lz;                                   // 1 .. 61
  unsigned long long top = (hi << lz) | (lo >> sh);         // bit 63 set
  top |= (lo << lz) != 0 ? 1ull : 0ull;                     // sticky bit, below the rounding bit
  return l8_ldexp((double)top, sh + sc);
}

// exact C' from its 16 symmetric residues, rounded to double and scaled by 2^sc.  S = sum_j t_j (M / m_j) with
// t_j = y_j (M / m_j)^-1 mod m_j < 256 is accumulated in four 32-bit limbs of M / m_j (one mad.wide.u32 each): every limb
// sum stays below 16 2^8 2^32 < 2^44, so the carries are propagated once after the loop.  S < 16 M; q = floor(S / M) is
// taken from the top 33 bits of S against the top limb of M, rounded up (q is exact or one too small), and fixed with one
// comparison.  Same x = S mod M as a 128-bit sum reduced after every step: the result is bit-identical.
__host__ __device__ __forceinline__ double l8_crt(const int (&y)[L8_NMOD], int sc) {
  const u128 M = ((u128)L8_M_HI << 64) | L8_M_LO;
  unsigned long long a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
  for (int j = 0; j < L8_NMOD; j++) {
    const L8Mod md = l8_mod(j);
    const unsigned yy = (unsigned)(y[j] < 0 ? y[j] + md.m : y[j]);
    const unsigned t = (yy * (unsigned)md.inv) % (unsigned)md.m;
    a0 += (unsigned long long)t * (unsigned)md.lo;
    a1 += (unsigned long long)t * (unsigned)(md.lo >> 32);
    a2 += (unsigned long long)t * (unsigned)md.hi;
    a3 += (unsigned long long)t * (unsigned)(md.hi >> 32);
  }
  a1 += a0 >> 32;
  a2 += a1 >> 32;
  a3 += a2 >> 32;   // S = a3 2^96 + (a2 mod 2^32) 2^64 + (a1 mod 2^32) 2^32 + (a0 mod 2^32), a3 < 2^33
  const unsigned long long q = a3 / ((L8_M_HI >> 32) + 1);
  u128 x = ((u128)a3 << 96) | ((u128)(a2 & 0xffffffffull) << 64) | ((a1 & 0xffffffffull) << 32) | (a0 & 0xffffffffull);
  x -= (u128)q * M;   // mod 2^128: the true difference is below 2 M < 2^128
  if (x >= M) x -= M;
  const bool neg = x > (M >> 1);
  return neg ? -l8_round(M - x, sc) : l8_round(x, sc);
}

// lower tiles (128 x 128) of an nb-block triangle in L2-aware order: bands of 8 block rows, cells of 8 x 8 tiles inside a
// band (band p has p + 1 cells, 32 p (p + 1) slots before it); the longest K (top band) first
__host__ __device__ inline int l8_slots(int nb) {
  const int B = (nb + 7) / 8;
  return 32 * B * (B + 1);
}

// ---------------------------------------------------------------- 1. conversion: one CTA per operand row
// Row i of the operand src[i][0, kw) (leading dimension lds), entries outside [k_lo(i), k_hi(i)) taken as zeros:
// k_lo(i) = 128 (i / 128) when lo_blk (upper block triangle: nothing left of the row's diagonal block is stored, the GEMM
// reads no k block left of it), else 0; k_hi(i) = 64 (i / 64 + 1) when hi64 (lower triangle at the 64-row granularity the
// DMMA tile engine reads), else kw.  Residues of plane j at R + j plane + i ldr + k.
__global__ void __launch_bounds__(256) k_l8_convert(const double* __restrict__ src, long long lds, int kw, int b, bool lo_blk,
                                                    bool hi64, int8_t* __restrict__ R, long long ldr, long long plane,
                                                    int* __restrict__ sexp) {
  const int i = blockIdx.x;
  const int k0 = lo_blk ? (i / 128) * 128 : 0;
  const int k1 = hi64 ? (i / 64 + 1) * 64 : kw;
  const double* row = src + (size_t)i * lds;
  __shared__ double red[8];
  double mx = 0.0;
  for (int k = k0 + threadIdx.x; k < k1; k += 256) mx = fmax(mx, fabs(row[k]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int w = 1; w < 8; w++) mx = fmax(mx, red[w]);
  int e = 0;
  if (mx > 0.0) frexp(mx, &e);      // mx < 2^e
  const int s = mx > 0.0 ? b - 1 - e : 0;
  if (threadIdx.x == 0) sexp[i] = s;
  int8_t* out = R + (size_t)i * ldr;
  for (int k = k0 + 8 * threadIdx.x; k < kw; k += 8 * 256) {
    const bool in = k < k1;   // k1 is a multiple of 64: the 8 entries lie wholly inside or outside the row's range
    unsigned long long a[8];
    bool neg[8];
#pragma unroll
    for (int v = 0; v < 8; v++) {
      const double x = in ? rint(ldexp(row[k + v], s)) : 0.0;   // exact scaling; |x| <= 2^(b-1) < 2^62
      neg[v] = x < 0.0;
      a[v] = (unsigned long long)fabs(x);
    }
#pragma unroll
    for (int j = 0; j < L8_NMOD; j++) {
      uint32_t w0 = 0, w1 = 0;
#pragma unroll
      for (int v = 0; v < 4; v++) w0 |= (uint32_t)(uint8_t)(int8_t)l8_residue(a[v], neg[v], j) << (8 * v);
#pragma unroll
      for (int v = 0; v < 4; v++) w1 |= (uint32_t)(uint8_t)(int8_t)l8_residue(a[4 + v], neg[4 + v], j) << (8 * v);
      *reinterpret_cast<uint2*>(out + j * plane + k) = make_uint2(w0, w1);
    }
  }
}

// ---------------------------------------------------------------- 2. modular GEMM (tcgen05, kind::i8)
__device__ __forceinline__ uint64_t l8_sdesc(uint32_t saddr) {
  // K-major operand, 128-byte swizzle (the TMA box layout): 8-row atoms of 128 B, 1024 B apart (SBO); version 1
  return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}
// instruction descriptor: S32 accumulator, signed 8-bit A and B, both K-major, N = 128, M = 128
constexpr uint32_t L8_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ void l8_mma(uint32_t tmem, uint64_t ad, uint64_t bd, uint32_t acc) {
  asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}"
               ::"r"(tmem), "l"(ad), "l"(bd), "r"(L8_IDESC), "r"(acc));
}
__device__ __forceinline__ void l8_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// one 128 x 128 output tile of plane j: C_j = sum over the k blocks kb0 .. kb0 + nk - 1 of A_j[rowA0 + 128) B_j[rowB0 + 128)'
// mod m_j (A_j, B_j: plane j of the two tensor maps), stored as int8 residues at dst (row stride lds)
__device__ __forceinline__ void l8_tile(const CUtensorMap* tmA, const CUtensorMap* tmB, int j, int rowA0, int rowB0, int kb0,
                                        int nk, int8_t* __restrict__ dst, long long lds) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + L8_STAGES * L8_STAGE_BYTES);
  uint64_t* empty = full + L8_STAGES;
  uint64_t* done = empty + L8_STAGES;
  uint32_t* tslot = (uint32_t*)(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < L8_STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(done, 1);
    fence_mbar_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;" ::"r"(smem_u32(tslot)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tslot;

  if (threadIdx.x == 0) {   // TMA producer
    for (int it = 0; it < nk; it++) {
      const int s = it % L8_STAGES;
      if (it >= L8_STAGES) mbar_wait(&empty[s], ((it / L8_STAGES) - 1) & 1);
      uint8_t* st = smem + s * L8_STAGE_BYTES;
      mbar_expect_tx(&full[s], L8_STAGE_BYTES);
      tma_load_3d(st, tmA, &full[s], (kb0 + it) * 128, rowA0, j);
      tma_load_3d(st + L8_TILE_BYTES, tmB, &full[s], (kb0 + it) * 128, rowB0, j);
    }
  } else if (threadIdx.x == 32) {   // MMA issuer
    for (int it = 0; it < nk; it++) {
      const int s = it % L8_STAGES;
      mbar_wait(&full[s], (it / L8_STAGES) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t sa = smem_u32(smem + s * L8_STAGE_BYTES);
      const uint64_t ad = l8_sdesc(sa), bd = l8_sdesc(sa + L8_TILE_BYTES);
#pragma unroll
      for (int kk = 0; kk < 4; kk++) l8_mma(tmem, ad + 2 * kk, bd + 2 * kk, (it | kk) != 0);   // +32 B of K per step
      l8_commit(&empty[s]);
    }
    l8_commit(done);
  }
  __syncwarp();

  // epilogue: thread t owns row 32 warp + lane of the tile (tensor-memory lane), 32 columns per load
  mbar_wait(done, 0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const int m = l8_mod(j).m;
  const double rinv = 1.0 / (double)m;
  dst += (size_t)(32 * warp + lane) * lds;
#pragma unroll 1
  for (int q = 0; q < 4; q++) {
    uint32_t v[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,"
        "%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(tmem + ((uint32_t)(32 * warp) << 16) + 32 * q));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    uint32_t w[8];
#pragma unroll
    for (int e = 0; e < 8; e++) w[e] = 0;
#pragma unroll
    for (int e = 0; e < 32; e++) {
      const int a = (int)v[e];
      const int res = a - (int)rint((double)a * rinv) * m;   // exact: a / m is never a half-integer (m odd)
      w[e >> 2] |= (uint32_t)(uint8_t)(int8_t)res << (8 * (e & 3));
    }
    uint4* o = reinterpret_cast<uint4*>(dst + 32 * q);
    o[0] = make_uint4(w[0], w[1], w[2], w[3]);
    o[1] = make_uint4(w[4], w[5], w[6], w[7]);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;" ::"r"(tmem));
  }
}

// LAUUM: grid = 16 * l8_slots(nb), modulus-major; modulus j is plane j of R (the third TMA coordinate) and of D
__global__ void __launch_bounds__(128, 2) k_l8_gemm(const __grid_constant__ CUtensorMap tmR, int nb, int8_t* __restrict__ R,
                                                    int8_t* __restrict__ D, long long ld) {
  const int slots = l8_slots(nb);
  const int j = blockIdx.x / slots, tile = blockIdx.x - j * slots;
  const int p = (isqrt_floor(4 * (tile >> 5) + 1) - 1) >> 1;
  const int rem = tile - 32 * p * (p + 1);
  const int i = 8 * p + ((rem & 63) >> 3), c = 8 * (rem >> 6) + (rem & 7);
  if (i >= nb || c > i) return;
  int8_t* dst = (i == c) ? D + (size_t)j * ld * 128 + (size_t)i * 128 * 128
                         : R + (size_t)j * ld * ld + (size_t)i * 128 * ld + (size_t)c * 128;
  l8_tile(&tmR, &tmR, j, i * 128, c * 128, i, nb - i, dst, i == c ? 128 : ld);   // k blocks i .. nb-1
}

// k ranges of k_l8_gemm_ab
enum { L8_KLOWER_B = 0, L8_KUPPER_A = 1, L8_KFULL_SYRK = 2 };

// C = A B' over ra x rb tiles (C residues [16][128 ra][128 rb]), the k blocks of tile (i, c) by kmode:
//   L8_KUPPER_A: [i, kb) (A upper block triangular, kb its block width); L8_KLOWER_B: [0, c + 1) (B lower block triangular);
//   L8_KFULL_SYRK: [0, kb), the lower tiles c <= i of a square product (rb = ra, A and B the same planes) only.
// Grid = 16 * 64 ceil(ra / 8) ceil(rb / 8): cells of 8 x 8 tiles, the longest K first (L8_KUPPER_A: row-major from the top;
// L8_KLOWER_B: column-major from the right); L8_KFULL_SYRK: 16 * l8_slots(ra), the band order of k_l8_gemm.
__global__ void __launch_bounds__(128, 2) k_l8_gemm_ab(const __grid_constant__ CUtensorMap tmA,
                                                       const __grid_constant__ CUtensorMap tmB, int ra, int rb, int kb,
                                                       int kmode, int8_t* __restrict__ C) {
  const long long ldc = 128LL * rb;
  if (kmode == L8_KFULL_SYRK) {
    const int slots = l8_slots(ra);
    const int j = blockIdx.x / slots, tile = blockIdx.x - j * slots;
    const int p = (isqrt_floor(4 * (tile >> 5) + 1) - 1) >> 1;
    const int rem = tile - 32 * p * (p + 1);
    const int i = 8 * p + ((rem & 63) >> 3), c = 8 * (rem >> 6) + (rem & 7);
    if (i >= ra || c > i) return;
    int8_t* dst = C + (size_t)j * 128 * ra * ldc + (size_t)i * 128 * ldc + (size_t)c * 128;
    l8_tile(&tmA, &tmB, j, i * 128, c * 128, 0, kb, dst, ldc);
    return;
  }
  const bool kupper = kmode == L8_KUPPER_A;
  const int cr = (ra + 7) / 8, cc = (rb + 7) / 8, slots = 64 * cr * cc;
  const int j = blockIdx.x / slots, tile = blockIdx.x - j * slots;
  const int cell = tile >> 6, w = tile & 63;
  const int i = 8 * (kupper ? cell / cc : cell % cr) + (w >> 3);
  const int c = kupper ? 8 * (cell % cc) + (w & 7) : 8 * (cc - 1 - cell / cr) + 7 - (w & 7);
  if (i >= ra || c < 0 || c >= rb) return;
  int8_t* dst = C + (size_t)j * 128 * ra * ldc + (size_t)i * 128 * ldc + (size_t)c * 128;
  if (kupper) l8_tile(&tmA, &tmB, j, i * 128, c * 128, i, kb - i, dst, ldc);
  else l8_tile(&tmA, &tmB, j, i * 128, c * 128, 0, c + 1, dst, ldc);
}

// ---------------------------------------------------------------- 3. reconstruction: one CTA per 128 x 128 tile
// out[r][c] = sign 2^-(sr[r] + sc[c]) C'[r][c] for the tile whose residues of plane j start at src + j plane (row stride ls);
// acc: out[r][c] += that instead (the product rounded once, then one FP64 addition)
__device__ __forceinline__ void l8_recon_tile(const int8_t* __restrict__ src, size_t plane, size_t ls,
                                              const int* __restrict__ sr, const int* __restrict__ sc, double sign,
                                              double* __restrict__ out, long long ldo, bool acc = false) {
  const int cq = 4 * (threadIdx.x & 31);
  const int sc0 = sc[cq], sc1 = sc[cq + 1], sc2 = sc[cq + 2], sc3 = sc[cq + 3];
#pragma unroll 1
  for (int rr = threadIdx.x >> 5; rr < 128; rr += 8) {
    const int8_t* p = src + (size_t)rr * ls + cq;
    int y[4][L8_NMOD];
#pragma unroll
    for (int j = 0; j < L8_NMOD; j++) {
      const uint32_t w = *reinterpret_cast<const uint32_t*>(p + j * plane);
#pragma unroll
      for (int v = 0; v < 4; v++) y[v][j] = (int)(int8_t)(w >> (8 * v));
    }
    const int s = sr[rr];
    double2 o0, o1;
    o0.x = sign * l8_crt(y[0], -(s + sc0));
    o0.y = sign * l8_crt(y[1], -(s + sc1));
    o1.x = sign * l8_crt(y[2], -(s + sc2));
    o1.y = sign * l8_crt(y[3], -(s + sc3));
    double* kp = out + (size_t)rr * ldo + cq;
    if (acc) {
      const double2 a0 = *reinterpret_cast<const double2*>(kp), a1 = *reinterpret_cast<const double2*>(kp + 2);
      o0.x = __dadd_rn(a0.x, o0.x); o0.y = __dadd_rn(a0.y, o0.y);
      o1.x = __dadd_rn(a1.x, o1.x); o1.y = __dadd_rn(a1.y, o1.y);
    }
    *reinterpret_cast<double2*>(kp) = o0;
    *reinterpret_cast<double2*>(kp + 2) = o1;
  }
}

// Kinv[r, c] for the lower block triangle (diagonal blocks in full), the region M_LAUUM writes
__global__ void __launch_bounds__(256) k_l8_recon(const int8_t* __restrict__ R, const int8_t* __restrict__ D, long long ld,
                                                  const int* __restrict__ sexp, double* __restrict__ K,
                                                  long long ldk) {
  const int t = blockIdx.x;
  int i = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while (i * (i + 1) / 2 > t) --i;
  while ((i + 1) * (i + 2) / 2 <= t) ++i;
  const int c = t - i * (i + 1) / 2;
  if (i == c) l8_recon_tile(D + (size_t)i * 128 * 128, (size_t)ld * 128, 128, sexp + i * 128, sexp + c * 128, 1.0,
                            K + (size_t)i * 128 * ldk + c * 128, ldk);
  else l8_recon_tile(R + (size_t)i * 128 * ld + c * 128, (size_t)ld * ld, ld, sexp + i * 128, sexp + c * 128, 1.0,
                     K + (size_t)i * 128 * ldk + c * 128, ldk);
}

// out[128 ra][128 rb] (leading dimension ldo) = sign C from the residues of k_l8_gemm_ab; one CTA per tile.
// syrk (the L8_KFULL_SYRK product, rb = ra): out += sign C on the lower tiles only (diagonal tiles in full), grid ra (ra + 1) / 2
__global__ void __launch_bounds__(256) k_l8_recon_ab(const int8_t* __restrict__ C, int ra, int rb, const int* __restrict__ sa,
                                                     const int* __restrict__ sb, double sign, double* __restrict__ out,
                                                     long long ldo, bool syrk) {
  int i, c;
  if (syrk) {
    const int t = blockIdx.x;
    i = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
    while (i * (i + 1) / 2 > t) --i;
    while ((i + 1) * (i + 2) / 2 <= t) ++i;
    c = t - i * (i + 1) / 2;
  } else {
    i = blockIdx.x / rb; c = blockIdx.x - i * rb;
  }
  const size_t ldc = (size_t)128 * rb;
  l8_recon_tile(C + (size_t)i * 128 * ldc + c * 128, (size_t)128 * ra * ldc, ldc, sa + i * 128, sb + c * 128, sign,
                out + (size_t)i * 128 * ldo + c * 128, ldo, syrk);
}

}  // namespace dgp
