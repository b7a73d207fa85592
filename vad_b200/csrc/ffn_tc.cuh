// ffn_tc.cuh -- Dense 39-64-32-16-3 (learning/ffn_trainer.py:104-116) on the 5th-gen tensor
// cores: tcgen05.mma kind::tf32, accumulators and activations in TMEM.
//
// Why tensor cores here (ncu, profiles/README.md r1a/r1b): with FP32 FFMAs the FFN block phase
// took 47 % of the fused kernel at 32 % FMA-pipe utilisation -- bound by delivering 5,104 weight
// operands per frame (LDCU) and by instruction fetch, not by math.  As an M=128-frame GEMM chain
// the same contraction is ~1 k CUDA-core instructions per frame (feature build + epilogues).
//
// Precision: logits must stay within 1e-3 of the float64 oracle, so every operand is split into
// two tf32 terms, x = x_hi + x_lo (x_hi = top 19 bits, x_lo = x - x_hi exactly), and each layer
// needs a_hi.b_hi + a_lo.b_hi + a_hi.b_lo (the dropped lo.lo term is <= 2^-20 relative), fp32
// accumulation in TMEM.  clock64 stamps showed every one of these tiny K=8 MMAs costs ~85 cycles
// whatever its N (latency-, not math-bound), so the B operand is stored as [B_hi | B_lo] (2N rows)
// and each k-step issues TWO instructions instead of three:
//     D'[0:2N] += a_hi . [B_hi | B_lo]      D'[0:N] += a_lo . B_hi
// and the epilogue adds the two halves D'[c] + D'[N + c].
//
// One tile = 128 frames = 128 threads (4 warps; warp w owns TMEM lanes 32 (w % 4) ..+31, thread =
// frame = lane).  TMEM map (256 columns per CTA, 2 CTAs per SM = all 512):
//   [  0,128)  A operand of the current layer: hi in [0,K), lo in [K,2K)   (K = 48, 64, 32, 16)
//   [128,256)  D1' (2 x 64)  -> later D2' [128,192) (2 x 32)
//   [192,224)  D3' (2 x 16)      [224,256)  D4' (2 x 16)
// Weights (B operand, 2N x K, K-major, SWIZZLE_NONE canonical layout: 8x16B core matrices, core
// (kc, nc) at (kc * 2N/8 + nc) * 128 B, rows [0,N) = hi, [N,2N) = lo, so SBO = 128 B and
// LBO = 2N/8 * 128 B) are prepared once on the host and arrive in shared memory by one TMA bulk copy.
#pragma once

#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "vad_core.cuh"

namespace vadb {

constexpr int kTcK1 = 48, kTcN1 = 64;   // 39 -> 48: two 24-column halves (coefficients 0-6 | 7-12), see tc_feat_col
// Layer-1 K order: feature (g, k) (g = 0 z, 1 d1, 2 d2; reference order g*13 + k) of coefficient pair q = k / 2,
// element e = k % 2 sits in column 6 q + 2 g + e for q < 4 and 24 + 6 (q - 4) + 2 g + e for q >= 4, so that the two
// threads sharing a frame each build the features of one range of coefficient pairs with packed arithmetic
// (vad_core.cuh window_features_pairs) and store one contiguous 24-column block whose fp16 column pairs are the
// packed results themselves.  Columns 40, 41 (the missing coefficient 13) and 42..47 are zero.
__host__ __device__ constexpr int tc_feat_col(int feat) {
  const int g = feat / 13, k = feat % 13, q = k / 2, e = k % 2;
  return q < 4 ? 6 * q + 2 * g + e : 24 + 6 * (q - 4) + 2 * g + e;
}
constexpr int kTcK2 = 64, kTcN2 = 32;
constexpr int kTcK3 = 32, kTcN3 = 16;
constexpr int kTcK4 = 16, kTcN4 = 16;   // 3 -> 16 (M = 128 needs N % 16 == 0)
constexpr int kTcBlk1 = kTcK1 * kTcN1 * 4, kTcBlk2 = kTcK2 * kTcN2 * 4, kTcBlk3 = kTcK3 * kTcN3 * 4,
              kTcBlk4 = kTcK4 * kTcN4 * 4;
constexpr int kTcOff1 = 0;  // each layer: one [kc][2N/8][8][4] block of 2 * kTcBlk bytes
constexpr int kTcOff2 = kTcOff1 + 2 * kTcBlk1;
constexpr int kTcOff3 = kTcOff2 + 2 * kTcBlk2;
constexpr int kTcOff4 = kTcOff3 + 2 * kTcBlk3;
constexpr int kTcBlobBytes = kTcOff4 + 2 * kTcBlk4;  // 47,104
constexpr int kTmemCols = 256;
constexpr int kTmA = 0, kTmD1 = 128, kTmD2 = 128, kTmD3 = 192, kTmD4 = 224;

// ---- host side: pack Keras (in,out) weights into the canonical hi/lo blob --------------------------
inline float tf32_hi(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  u &= 0xFFFFE000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}
inline void tc_pack_layer(const float* W /*[k_real][n_real]*/, int k_real, int n_real, int K, int N, float* blk,
                          bool permute_features = false) {
  for (int i = 0; i < 2 * K * N; ++i) blk[i] = 0.0f;
  for (int n = 0; n < n_real; ++n)
    for (int kk = 0; kk < k_real; ++kk) {
      const float w = W[kk * n_real + n];
      const int k = permute_features ? tc_feat_col(kk) : kk;
      const float hi = tf32_hi(w);
      const int ihi = ((k / 4) * (2 * N / 8) + (n / 8)) * 32 + (n % 8) * 4 + (k % 4);
      const int ilo = ((k / 4) * (2 * N / 8) + ((N + n) / 8)) * 32 + ((N + n) % 8) * 4 + (k % 4);
      blk[ihi] = hi;
      blk[ilo] = w - hi;
    }
}
inline void tc_pack_weights(const FfnParams& p, unsigned char* blob /*kTcBlobBytes*/) {
  tc_pack_layer(p.W1, kNFeat, kH1, kTcK1, kTcN1, reinterpret_cast<float*>(blob + kTcOff1), true);
  tc_pack_layer(p.W2, kH1, kH2, kTcK2, kTcN2, reinterpret_cast<float*>(blob + kTcOff2));
  tc_pack_layer(p.W3, kH2, kH3, kTcK3, kTcN3, reinterpret_cast<float*>(blob + kTcOff3));
  tc_pack_layer(p.W4, kH3, kNCls, kTcK4, kTcN4, reinterpret_cast<float*>(blob + kTcOff4));
}

// ---- fp16 hi/lo operand path (kind::f16, K = 16 per instruction: half the MMAs of the tf32 path) -------
// Same three-product scheme with x = x_hi + x_lo in fp16 (11-bit significands, like tf32).  fp16's narrow
// exponent range is handled statically: every layer's weights are scaled by a power of two sw_l into
// [8192, 16384), every layer's input activations by a power of two sa_l chosen from a rigorous bound on
// their magnitude (features are bounded by the MFCC range, hidden activations by sum |W| x bound), so no
// operand can overflow; the epilogue multiplies D by 1 / (sw_l sa_l) (exact).  A handle whose weights
// would need an absurd scale keeps the tf32 path.
constexpr int kTc16Blk1 = kTcK1 * kTcN1 * 2, kTc16Blk2 = kTcK2 * kTcN2 * 2, kTc16Blk3 = kTcK3 * kTcN3 * 2,
              kTc16Blk4 = kTcK4 * kTcN4 * 2;          // bytes of one [K][N] fp16 block; hi | lo doubles it
constexpr int kTc16Off1 = 0;
constexpr int kTc16Off2 = kTc16Off1 + 2 * kTc16Blk1;
constexpr int kTc16Off3 = kTc16Off2 + 2 * kTc16Blk2;
constexpr int kTc16Off4 = kTc16Off3 + 2 * kTc16Blk3;
constexpr int kTc16BlobBytes = kTc16Off4 + 2 * kTc16Blk4;  // 23,552
// rigorous feature bounds (vad_core.cuh window_features): |z| <= 2 (n = 5), |c| <= 1353 (|log2 E| <= 52 times the
// largest row sum of the folded DCT matrix), so |d1| <= 2706 and |d2| <= 5412 in either feature recipe
constexpr float kFeatBoundZ = 1353.0f, kFeatBoundD1 = 2706.0f, kFeatBoundD2 = 5416.0f;

inline uint16_t f32_to_f16_rn(float f) {  // round-to-nearest-even, subnormals, no NaN inputs expected
  uint32_t x;
  memcpy(&x, &f, 4);
  const uint32_t sign = (x >> 16) & 0x8000u;
  x &= 0x7FFFFFFFu;
  if (x >= 0x47800000u) return static_cast<uint16_t>(sign | 0x7C00u);  // overflow -> inf (never: scales prevent it)
  if (x < 0x38800000u) {                                               // subnormal half (or zero)
    if (x < 0x33000000u) return static_cast<uint16_t>(sign);
    const uint32_t mant = (x & 0x7FFFFFu) | 0x800000u;
    const int shift = 126 - static_cast<int>(x >> 23);                // 14 .. 24
    uint32_t h = mant >> shift;
    const uint32_t rem = mant & ((1u << shift) - 1u), half = 1u << (shift - 1);
    if (rem > half || (rem == half && (h & 1u))) ++h;
    return static_cast<uint16_t>(sign | h);
  }
  uint32_t h = ((x >> 23) - 112u) << 10 | ((x >> 13) & 0x3FFu);
  const uint32_t rem = x & 0x1FFFu;
  if (rem > 0x1000u || (rem == 0x1000u && (h & 1u))) ++h;
  return static_cast<uint16_t>(sign | h);
}
inline float f16_to_f32(uint16_t h) {
  const uint32_t sign = (h & 0x8000u) << 16, e = (h >> 10) & 0x1Fu, m = h & 0x3FFu;
  if (e == 0) return (sign ? -1.0f : 1.0f) * std::ldexp(static_cast<float>(m), -24);
  uint32_t x = sign | ((e + 112u) << 23) | (m << 13);
  float f;
  memcpy(&f, &x, 4);
  return f;
}
inline void tc16_pack_layer(const float* W /*[k_real][n_real]*/, int k_real, int n_real, int K, int N, float sw,
                            uint16_t* blk, bool permute_features = false) {
  for (int i = 0; i < 2 * K * N; ++i) blk[i] = 0;
  for (int n = 0; n < n_real; ++n)
    for (int kk = 0; kk < k_real; ++kk) {
      const float w = W[kk * n_real + n] * sw;
      const int k = permute_features ? tc_feat_col(kk) : kk;
      const uint16_t hi = f32_to_f16_rn(w);
      const uint16_t lo = f32_to_f16_rn(w - f16_to_f32(hi));
      const int ihi = ((k / 8) * (2 * N / 8) + (n / 8)) * 64 + (n % 8) * 8 + (k % 8);
      const int ilo = ((k / 8) * (2 * N / 8) + ((N + n) / 8)) * 64 + ((N + n) % 8) * 8 + (k % 8);
      blk[ihi] = hi;
      blk[ilo] = lo;
    }
}
// Chooses the scales, packs the blob, fills bias.post / bias.pre.  Returns false if a scale exponent is
// out of the range the scheme was validated for (the handle then keeps the tf32 path).
inline bool tc16_pack_weights(const FfnParams& p, unsigned char* blob /*kTc16BlobBytes*/, FfnBias& fb) {
  const float* W[4] = {p.W1, p.W2, p.W3, p.W4};
  const float* B[4] = {p.b1, p.b2, p.b3, p.b4};
  const int kin[4] = {kNFeat, kH1, kH2, kH3}, nout[4] = {kH1, kH2, kH3, kNCls};
  const int Kp[4] = {kTcK1, kTcK2, kTcK3, kTcK4}, Np[4] = {kTcN1, kTcN2, kTcN3, kTcN4};
  const int off[4] = {kTc16Off1, kTc16Off2, kTc16Off3, kTc16Off4};
  std::vector<double> bound(kNFeat);
  for (int i = 0; i < kNFeat; ++i) bound[i] = i < kNCep ? kFeatBoundZ : i < 2 * kNCep ? kFeatBoundD1 : kFeatBoundD2;
  for (int l = 0; l < 4; ++l) {
    double amax = 0.0, wmax = 0.0;
    for (double b : bound) amax = std::max(amax, b);
    for (int i = 0; i < kin[l] * nout[l]; ++i) wmax = std::max(wmax, static_cast<double>(std::fabs(W[l][i])));
    if (!(amax < 1e30) || !(wmax < 1e30)) return false;
    // activations into (-32768, 32768), weights into [8192, 16384)
    const int ea = amax > 32000.0 ? static_cast<int>(std::ceil(std::log2(amax / 32000.0))) : 0;
    const int ew = wmax > 0.0 ? static_cast<int>(std::floor(std::log2(16000.0 / wmax))) : 0;
    if (ea > 60 || ew > 60 || ew < -60) return false;
    const float sa = std::ldexp(1.0f, -ea), sw = std::ldexp(1.0f, ew);
    if (l == 0 && ea != 0) return false;  // the feature bounds keep layer 1's activations unscaled (pre[0] == 1)
    fb.pre[l] = sa;
    fb.post[l] = std::ldexp(1.0f, ea - ew);
    tc16_pack_layer(W[l], kin[l], nout[l], Kp[l], Np[l], sw, reinterpret_cast<uint16_t*>(blob + off[l]), l == 0);
    std::vector<double> nb(nout[l]);
    for (int j = 0; j < nout[l]; ++j) {
      double s = std::fabs(static_cast<double>(B[l][j]));
      for (int i = 0; i < kin[l]; ++i) s += std::fabs(static_cast<double>(W[l][i * nout[l] + j])) * bound[i];
      nb[j] = s;
    }
    bound = nb;
  }
  for (int l = 0; l < 3; ++l) fb.postp[l] = fb.post[l] * fb.pre[l + 1];
  fb.postp[3] = fb.post[3];
  for (int j = 0; j < kH1; ++j) fb.c1[j] = p.b1[j] * fb.pre[1];
  for (int j = 0; j < kH2; ++j) fb.c2[j] = p.b2[j] * fb.pre[2];
  for (int j = 0; j < kH3; ++j) fb.c3[j] = p.b3[j] * fb.pre[3];
  return true;
}

#if defined(__CUDACC__)
// ---- PTX wrappers ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(
          taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
               "r"(v[2]), "r"(v[3])
               : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem]^T, M = 128, kind::tf32 (K = 8 per instruction); one thread issues.
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {  // implies tcgen05.fence::before_thread_sync
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ bool tc_mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(tc_smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void tc_mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!tc_mbar_try_wait(bar, parity)) {
  }
}

// K-major, SWIZZLE_NONE shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout)
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;  // descriptor version for sm_100
  return d;
}
__host__ __device__ constexpr uint32_t tc_idesc(int n) {
  return (1u << 4) /* D = f32 */ | (2u << 7) /* A = tf32 */ | (2u << 10) /* B = tf32 */ |
         (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(128 >> 4) << 24);
}

// One layer: 2 MMAs per k-step (a_hi . [B_hi | B_lo] into 2N columns, a_lo . B_hi into the first N);
// executed by ONE thread.
template <int K, int N>
__device__ __forceinline__ void tc_issue_layer(uint32_t tm_base, uint32_t d_col, uint32_t w_smem, uint64_t* done_bar) {
  constexpr uint32_t lbo = (2 * N / 8) * 128, sbo = 128;
  constexpr uint32_t idesc_2n = tc_idesc(2 * N), idesc_n = tc_idesc(N);
  const uint32_t a_hi = tm_base + kTmA, a_lo = tm_base + kTmA + K, d = tm_base + d_col;
#pragma unroll
  for (int j = 0; j < K / 8; ++j) {
    const uint64_t b = tc_smem_desc(w_smem + 2 * j * lbo, lbo, sbo);
    umma_tf32_ts(d, a_hi + 8 * j, b, idesc_2n, j > 0 ? 1u : 0u);
    umma_tf32_ts(d, a_lo + 8 * j, b, idesc_n, 1u);
  }
  umma_commit(done_bar);
}

__device__ __forceinline__ void tc_split(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xFFFFE000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}

// Epilogue of a hidden layer: D (NOUT fp32 columns at d_col) -> + bias, ReLU, hi/lo split -> A operand
// of the next layer (hi at [0,NOUT), lo at [NOUT,2 NOUT)).  With HALVES = 2 two threads share a frame
// (warp w and w + 4 own the same TMEM lane quarter) and each converts NOUT/2 columns.
template <int NOUT, int HALVES>
__device__ __forceinline__ void tc_hidden_epilogue(uint32_t tl, uint32_t d_col, const float* bias, int hidx) {
  constexpr int W = NOUT / HALVES;         // columns per thread: 64, 32, 16 or 8
  constexpr int CH = W >= 16 ? 16 : 8;     // chunk width
  const int base = hidx * W;
#pragma unroll
  for (int c0 = 0; c0 < W; c0 += CH) {
    uint32_t v[CH], u[CH], hi[CH], lo[CH];
    if constexpr (CH == 16) {
      tmem_ld16(tl + d_col + base + c0, v);           // a . B_hi
      tmem_ld16(tl + d_col + NOUT + base + c0, u);    // a_hi . B_lo
    } else {
      tmem_ld8(tl + d_col + base + c0, v);
      tmem_ld8(tl + d_col + NOUT + base + c0, u);
    }
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      const float a = fmaxf((__uint_as_float(v[i]) + __uint_as_float(u[i])) + bias[base + c0 + i], 0.0f);
      tc_split(a, hi[i], lo[i]);
    }
    if constexpr (CH == 16) {
      tmem_st16(tl + kTmA + base + c0, hi);
      tmem_st16(tl + kTmA + NOUT + base + c0, lo);
    } else {
      tmem_st8(tl + kTmA + base + c0, hi);
      tmem_st8(tl + kTmA + NOUT + base + c0, lo);
    }
  }
  tmem_wait_st();
}

template <int HALVES>
__device__ __forceinline__ void tc_bar() {
  if constexpr (HALVES == 2) asm volatile("bar.sync 1, 256;" ::: "memory");
  else asm volatile("bar.sync 1, 128;" ::: "memory");
}

// Store 24 layer-1 A columns (one half: hidx = 0 -> columns [0,24), 1 -> [24,48)) of this thread's frame.
__device__ __forceinline__ void tc_store_a1_half(uint32_t tl, int hidx, const float (&xl)[24]) {
  uint32_t hi[16], lo[16], hi8[8], lo8[8];
#pragma unroll
  for (int i = 0; i < 16; ++i) tc_split(xl[i], hi[i], lo[i]);
#pragma unroll
  for (int i = 0; i < 8; ++i) tc_split(xl[16 + i], hi8[i], lo8[i]);
  const uint32_t b = tl + kTmA + 24 * hidx;
  tmem_st16(b, hi);
  tmem_st8(b + 16, hi8);
  tmem_st16(b + kTcK1, lo);
  tmem_st8(b + kTcK1 + 16, lo8);
}

// The whole FFN for one 128-frame tile, executed by 128 * HALVES threads.  Thread (wq = warp % 4, lane)
// owns TMEM lane 32 wq + lane = one frame; with HALVES = 2 the threads of warp w and w + 4 share that
// frame (hidx = warp / 4): each has already stored its half of the layer-1 A operand
// (tc_store_a1_half) and they split every later layer's columns.  With HALVES = 1 the single thread
// stored both halves.  Logits are returned to hidx == 0.  w_smem: shared-memory address of the weight
// blob (already landed); mma_bar: mbarrier (count 1) whose current phase parity is `par` (4 phases).
template <int HALVES>
__device__ __forceinline__ uint32_t ffn_tc_tile(const FfnBias& fb, float (&logit)[kNCls], uint32_t tm_base, int wq, int hidx,
                                                bool is_issuer, uint32_t w_smem, uint64_t* mma_bar, uint32_t par,
                                                long long* ts = nullptr, int dbg = 0) {
  const uint32_t tl = tm_base + (static_cast<uint32_t>(32 * wq) << 16);
#define VADB_TS(i) do { if (ts) ts[i] = clock64(); } while (0)
  tmem_wait_st();
  tc_fence_before();
  tc_bar<HALVES>();
  VADB_TS(3);
  if (is_issuer && !(dbg & 32)) {
    tc_fence_after();
    tc_issue_layer<kTcK1, kTcN1>(tm_base, kTmD1, w_smem + kTcOff1, mma_bar);
  }
  VADB_TS(4);
  if (!(dbg & 32)) { tc_mbar_wait(mma_bar, par); par ^= 1u; }
  tc_fence_after();
  VADB_TS(5);
  if (!(dbg & 128)) tc_hidden_epilogue<kTcN1, HALVES>(tl, kTmD1, fb.b1, hidx);
  VADB_TS(6);
  tc_fence_before();
  tc_bar<HALVES>();
  if (is_issuer && !(dbg & 32)) {
    tc_fence_after();
    tc_issue_layer<kTcK2, kTcN2>(tm_base, kTmD2, w_smem + kTcOff2, mma_bar);
  }
  VADB_TS(7);
  if (!(dbg & 32)) { tc_mbar_wait(mma_bar, par); par ^= 1u; }
  tc_fence_after();
  VADB_TS(8);
  if (!(dbg & 128)) tc_hidden_epilogue<kTcN2, HALVES>(tl, kTmD2, fb.b2, hidx);
  VADB_TS(9);
  tc_fence_before();
  tc_bar<HALVES>();
  if (is_issuer && !(dbg & 32)) {
    tc_fence_after();
    tc_issue_layer<kTcK3, kTcN3>(tm_base, kTmD3, w_smem + kTcOff3, mma_bar);
  }
  VADB_TS(10);
  if (!(dbg & 32)) { tc_mbar_wait(mma_bar, par); par ^= 1u; }
  tc_fence_after();
  VADB_TS(11);
  if (!(dbg & 128)) tc_hidden_epilogue<kTcN3, HALVES>(tl, kTmD3, fb.b3, hidx);
  VADB_TS(12);
  tc_fence_before();
  tc_bar<HALVES>();
  if (is_issuer && !(dbg & 32)) {
    tc_fence_after();
    tc_issue_layer<kTcK4, kTcN4>(tm_base, kTmD4, w_smem + kTcOff4, mma_bar);
  }
  VADB_TS(13);
  if (!(dbg & 32)) { tc_mbar_wait(mma_bar, par); par ^= 1u; }
  tc_fence_after();
  VADB_TS(14);
  if (hidx == 0) {
    uint32_t v[8], u[8];
    tmem_ld8(tl + kTmD4, v);
    tmem_ld8(tl + kTmD4 + kTcN4, u);
    tmem_wait_ld();
#pragma unroll
    for (int o = 0; o < kNCls; ++o) logit[o] = (__uint_as_float(v[o]) + __uint_as_float(u[o])) + fb.b4[o];
  }
  tc_fence_before();  // the next tile's tcgen05.st must not overtake these loads
  VADB_TS(15);
#undef VADB_TS
  return par;
}

// ======================================= fp16 hi/lo variant ===========================================
// A operand in TMEM: two fp16 per 32-bit column (element 2c in the low half), hi parts in columns
// [0, K/2), lo parts in [K/2, K).  One instruction covers K = 16 = 8 columns.
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__host__ __device__ constexpr uint32_t tc16_idesc(int n) {
  return (1u << 4) /* D = f32; A = B = f16 (format 0), both K-major */ | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(128 >> 4) << 24);
}
// (x0, x1) -> one 32-bit word of hi parts and one of lo parts (element 0 in the low half); the residual is one FADD2
__device__ __forceinline__ void tc16_split2(f2 x, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(x.x, x.y);
  const float2 hf = __half22float2(h);
  const f2 r = vsub(x, mk2(hf.x, hf.y));
  const __half2 l = __floats2half2_rn(r.x, r.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
// Epilogue of a hidden layer on the 2N scheme: D (NOUT fp32 columns at d_col, second half NOUT further) -> x (post-scale
// x next layer's pre-scale), + scaled bias, ReLU, fp16 hi/lo split -> A operand of the next layer.  Column pairs are
// processed with packed fp32 arithmetic (tcgen05.ld delivers neighbouring columns in neighbouring registers).  One
// thread per frame.  cbias: bias x next pre-scale (FfnBias::c1..c3), postp: FfnBias::postp[l].
template <int NOUT>
__device__ __forceinline__ void tc16_hidden_epilogue(uint32_t tl, uint32_t d_col, const float* cbias, float postp) {
  static_assert(NOUT % 16 == 0, "16-column chunks");
#pragma unroll
  for (int c0 = 0; c0 < NOUT; c0 += 16) {
    uint32_t v[16], u[16], hi[8], lo[8];
    tmem_ld16(tl + d_col + c0, v);
    tmem_ld16(tl + d_col + NOUT + c0, u);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 16; i += 2) {
      const f2 d = vadd(mk2(__uint_as_float(v[i]), __uint_as_float(v[i + 1])),
                        mk2(__uint_as_float(u[i]), __uint_as_float(u[i + 1])));
      f2 a = vfma(d, mk2(postp, postp), mk2(cbias[c0 + i], cbias[c0 + i + 1]));
      a.x = fmaxf(a.x, 0.0f);
      a.y = fmaxf(a.y, 0.0f);
      tc16_split2(a, hi[i / 2], lo[i / 2]);
    }
    tmem_st8(tl + kTmA + c0 / 2, hi);
    tmem_st8(tl + kTmA + NOUT / 2 + c0 / 2, lo);
  }
  tmem_wait_st();
}
// 24 layer-1 A columns of one half (features of coefficient pairs 0-3 / 4-6, unscaled: FfnBias::pre[0] == 1)
// -> 12 + 12 packed columns.
__device__ __forceinline__ void tc16_store_a1_half(uint32_t tl, int hidx, const float (&xl)[24]) {
  uint32_t hi[8], lo[8], hi4[4], lo4[4];
#pragma unroll
  for (int i = 0; i < 8; ++i) tc16_split2(mk2(xl[2 * i], xl[2 * i + 1]), hi[i], lo[i]);
#pragma unroll
  for (int i = 0; i < 4; ++i) tc16_split2(mk2(xl[16 + 2 * i], xl[17 + 2 * i]), hi4[i], lo4[i]);
  const uint32_t b = tl + kTmA + 12 * hidx;
  tmem_st8(b, hi);
  tmem_st4(b + 8, hi4);
  tmem_st8(b + kTcK1 / 2, lo);
  tmem_st4(b + kTcK1 / 2 + 8, lo4);
}

// ================================ fp16 tiles: one or two per CTA ======================================
// TILES = 2 is the fused kernel's block phase: 256 frames, thread = frame, warp w serves tile w / 4 on TMEM lane quarter
// w % 4.  TILES = 1 is ffn_tc_rows_kernel's 128-row tile on warps 0-3.  Tile t owns columns [128 t, 128 t + 128) of the
// CTA's 256: the A operand (packed hi | lo, at most 32 + 32 columns) in the first 64, the fp32 accumulators in the last
// 64.  Layer 1's 2N scheme would need 2 x 64 accumulator columns, so layer 1 accumulates all three products into ONE
// 64-column accumulator, per k-step in the order a_hi.B_hi, a_hi.B_lo, a_lo.B_hi (B_lo is the same descriptor N/8 core
// matrices further on: the blob is unchanged).  Layers 2-4 keep the 2N scheme (2 x 32, 2 x 16 and 2 x 16 columns fit);
// with one accumulator they ran 0.7 % slower.  The fused block phase's fixed costs (barriers, synchronous DCT, blob
// copy, four MMA round trips) are paid once per 256 frames instead of once per 128.  Each epilogue overwrites A only
// after that layer's MMAs have completed.
constexpr int kTm2Tile = 128;                                      // TMEM columns per tile
constexpr int kTm2D1 = 64, kTm2D2 = 64, kTm2D3 = 64, kTm2D4 = 96;  // accumulators, relative to the tile
static_assert(2 * kTm2Tile == kTmemCols && kTm2D1 + kTcN1 <= kTm2Tile && kTm2D2 + 2 * kTcN2 <= kTm2Tile &&
              kTm2D4 + 2 * kTcN4 <= kTm2Tile && kTcK2 <= kTm2D1, "two tiles share the CTA's TMEM allocation");

// One layer of tile 0 and, if two_tiles, tile 1, interleaved MMA by MMA so that the tensor pipe always has an
// independent instruction between two that accumulate into the same columns; one commit.  Executed by ONE thread.
// ONE_ACC: a_hi.B_hi, a_hi.B_lo, a_lo.B_hi into N columns; otherwise a_hi . [B_hi | B_lo] into 2N columns and
// a_lo . B_hi into the first N.
template <int K, int N, bool ONE_ACC>
__device__ __forceinline__ void tc16_issue_layer(uint32_t tm_base, uint32_t d_col, uint32_t w_smem, bool two_tiles,
                                                 uint64_t* done_bar) {
  constexpr uint32_t lbo = (2 * N / 8) * 128, sbo = 128, lo_off = (N / 8) * 128;
  constexpr int kMmas = ONE_ACC ? 3 : 2;
#pragma unroll
  for (int j = 0; j < K / 16; ++j) {
    const uint32_t b = w_smem + 2 * j * lbo;
    const uint64_t b_hi = tc_smem_desc(b, lbo, sbo), b_lo = tc_smem_desc(b + lo_off, lbo, sbo);
#pragma unroll
    for (int m = 0; m < kMmas; ++m) {
      const uint32_t a_col = kTmA + (m == kMmas - 1 ? K / 2 : 0) + 8 * j;   // the last product takes a_lo
      const uint64_t bd = (ONE_ACC && m == 1) ? b_lo : b_hi;
      const uint32_t idesc = (!ONE_ACC && m == 0) ? tc16_idesc(2 * N) : tc16_idesc(N);
      const uint32_t acc = (j > 0 || m > 0) ? 1u : 0u;
      umma_f16_ts(tm_base + d_col, tm_base + a_col, bd, idesc, acc);
      if (two_tiles) umma_f16_ts(tm_base + kTm2Tile + d_col, tm_base + kTm2Tile + a_col, bd, idesc, acc);
    }
  }
  umma_commit(done_bar);
}
// Epilogue of layer 1 on its single accumulator: D (NOUT fp32 columns at d_col) -> x postp + cbias, ReLU, fp16
// hi/lo split -> A operand of the next layer (hi in [0, NOUT/2), lo in [NOUT/2, NOUT)).  One thread per frame.
template <int NOUT>
__device__ __forceinline__ void tc16_epilogue_1acc(uint32_t tl, uint32_t d_col, const float* cbias, float postp) {
#pragma unroll
  for (int c0 = 0; c0 < NOUT; c0 += 16) {
    uint32_t v[16], hi[8], lo[8];
    tmem_ld16(tl + d_col + c0, v);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 16; i += 2) {
      f2 a = vfma(mk2(__uint_as_float(v[i]), __uint_as_float(v[i + 1])), mk2(postp, postp),
                  mk2(cbias[c0 + i], cbias[c0 + i + 1]));
      a.x = fmaxf(a.x, 0.0f);
      a.y = fmaxf(a.y, 0.0f);
      tc16_split2(a, hi[i / 2], lo[i / 2]);
    }
    tmem_st8(tl + kTmA + c0 / 2, hi);
    tmem_st8(tl + kTmA + NOUT / 2 + c0 / 2, lo);
  }
  tmem_wait_st();
}
// The whole FFN for TILES 128-frame tiles, executed by 128 TILES threads; each thread has stored both halves of its
// frame's layer-1 A operand (tc16_store_a1_half at tl = ffn_tc16_tile_lane(...)) and gets its frame's logits.
// two_tiles (TILES = 2 only, block-uniform) false: tile 1 holds no valid frame and its MMAs are not issued (the
// epilogues of warps 4-7 then work on stale columns and their logits are meaningless).  w_smem: shared-memory address
// of the fp16 weight blob (already landed); mma_bar: mbarrier (count 1) whose current phase parity is `par` (4
// phases).  ts: clock64 stamps 3..15 (timing experiments only, same stages as ffn_tc_tile's).
__device__ __forceinline__ uint32_t ffn_tc16_tile_lane(uint32_t tm_base, int warp) {
  return tm_base + kTm2Tile * static_cast<uint32_t>(warp >> 2) + (static_cast<uint32_t>(32 * (warp & 3)) << 16);
}
template <int TILES>
__device__ __forceinline__ uint32_t ffn_tc16_tile(const FfnBias& fb, float (&logit)[kNCls], uint32_t tm_base, int warp,
                                                  bool two_tiles, bool is_issuer, uint32_t w_smem, uint64_t* mma_bar,
                                                  uint32_t par, long long* ts = nullptr) {
  static_assert(TILES == 1 || TILES == 2, "one or two tiles");
  const uint32_t tl = ffn_tc16_tile_lane(tm_base, warp);
  two_tiles = TILES == 2 && two_tiles;
#define VADB_TS(i) do { if (ts) ts[i] = clock64(); } while (0)
  tmem_wait_st();
  tc_fence_before();
  tc_bar<TILES>();
  VADB_TS(3);
  if (is_issuer) {
    tc_fence_after();
    tc16_issue_layer<kTcK1, kTcN1, true>(tm_base, kTm2D1, w_smem + kTc16Off1, two_tiles, mma_bar);
  }
  VADB_TS(4);
  tc_mbar_wait(mma_bar, par); par ^= 1u;
  tc_fence_after();
  VADB_TS(5);
  tc16_epilogue_1acc<kTcN1>(tl, kTm2D1, fb.c1, fb.postp[0]);
  VADB_TS(6);
  tc_fence_before();
  tc_bar<TILES>();
  if (is_issuer) {
    tc_fence_after();
    tc16_issue_layer<kTcK2, kTcN2, false>(tm_base, kTm2D2, w_smem + kTc16Off2, two_tiles, mma_bar);
  }
  VADB_TS(7);
  tc_mbar_wait(mma_bar, par); par ^= 1u;
  tc_fence_after();
  VADB_TS(8);
  tc16_hidden_epilogue<kTcN2>(tl, kTm2D2, fb.c2, fb.postp[1]);
  VADB_TS(9);
  tc_fence_before();
  tc_bar<TILES>();
  if (is_issuer) {
    tc_fence_after();
    tc16_issue_layer<kTcK3, kTcN3, false>(tm_base, kTm2D3, w_smem + kTc16Off3, two_tiles, mma_bar);
  }
  VADB_TS(10);
  tc_mbar_wait(mma_bar, par); par ^= 1u;
  tc_fence_after();
  VADB_TS(11);
  tc16_hidden_epilogue<kTcN3>(tl, kTm2D3, fb.c3, fb.postp[2]);
  VADB_TS(12);
  tc_fence_before();
  tc_bar<TILES>();
  if (is_issuer) {
    tc_fence_after();
    tc16_issue_layer<kTcK4, kTcN4, false>(tm_base, kTm2D4, w_smem + kTc16Off4, two_tiles, mma_bar);
  }
  VADB_TS(13);
  tc_mbar_wait(mma_bar, par); par ^= 1u;
  tc_fence_after();
  VADB_TS(14);
  {
    uint32_t v[8], u[8];
    tmem_ld8(tl + kTm2D4, v);
    tmem_ld8(tl + kTm2D4 + kTcN4, u);
    tmem_wait_ld();
#pragma unroll
    for (int o = 0; o < kNCls; ++o) logit[o] = fmaf(__uint_as_float(v[o]) + __uint_as_float(u[o]), fb.post[3], fb.b4[o]);
  }
  tc_fence_before();  // the next tile's tcgen05.st must not overtake these loads
  VADB_TS(15);
#undef VADB_TS
  return par;
}
#endif  // __CUDACC__

}  // namespace vadb
