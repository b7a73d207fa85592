// vad_core.cuh -- per-thread arithmetic of the fused MFCC + FFN VAD path (sm_100a).
//
// Everything here is plain C++17 marked __host__ __device__, so the same code is
//   * inlined into the CUDA kernels of vad_kernels.cu (the product), and
//   * compiled by g++ into tests/emul/ (a host emulation of the kernels' thread/lane
//     dataflow, used only by the CPU test-suite to validate index math and fp32 accuracy
//     where no GPU is available).  It is NOT a CPU fallback: the C ABI never calls it on
//     the host.
//
// Reference semantics restated here (paths relative to /root/reference):
//   mfcc.py:59-61   get_spec_mag      |FFT512(frame ++ zeros)[0:256] / 512|^2, rectangular window
//   mfcc.py:72-78   get_mfcc_from_spec  fbank dot, ==0 -> eps, log10, DCT-II ortho [:13], lifter
//   realtime_analysis/sklearn_analyser.py:52-69,103-107   5-frame window features
//   dataset/file_processing.py:51-66                     dataset-mode deltas
//   learning/ffn_trainer.py:104-116                      Dense 39-64-32-16-3
//
// FFT layout (one 400-sample real frame -> 256 power bins), 16 threads per frame:
//   z[n] = x[2n] + i x[2n+1], n < 256 (n >= 200 is zero padding); Z = FFT256(z) as 16 x 16
//   Cooley-Tukey:  pass 1: thread t holds z[t + 16 j], DFT16 over j (inputs j >= 13 are
//   structurally zero and pruned), times W256^(t k1); 16x16 transpose through shared memory;
//   pass 2: thread k1 DFT16 over n2 -> Z[k1 + 16 k2].  Real-FFT split: X[k] = (E + W512^k O)/2
//   with E = Z[k] + conj Z[256-k], O = -i (Z[k] - conj Z[256-k]); Z[256-k] lives in the
//   partner thread (16 - k1) & 15 and arrives by warp shuffle.  Power is kept as |2X|^2;
//   the 2^-20 = 1/(4*512^2) scale is folded into the mel weights.
#pragma once

#include <cmath>
#include <cstdint>
#include <type_traits>
#include <utility>

#include "vad_tables.h"

#if defined(__CUDACC__)
#define VADB_HD __host__ __device__ __forceinline__
#define VADB_CONSTANT __constant__
#else
#define VADB_HD inline
#define VADB_CONSTANT static
#endif

namespace vadb {

constexpr int kFrame = 400;      // config.py:21 FRAME_SIZE
constexpr int kHop = 160;        // config.py:22 FRAME_STEP
constexpr int kFftN = 512;       // config.py:27 FFT_N
constexpr int kBins = 256;       // fft_n / 2 (mfcc.py:61)
constexpr int kNMel = 26;        // config.py:25
constexpr int kNCep = 13;        // config.py:26
constexpr int kNFeat = 39;       // 13 x (mfcc, d1, d2)
constexpr int kH1 = 64, kH2 = 32, kH3 = 16, kNCls = 3;  // ffn_trainer.py:108-115

// ---- parameter blocks ---------------------------------------------------------------------------
// Mel / DCT tables depend only on the (single, compiled-in) reference configuration, so every
// handle uploads bit-identical content: the __constant__ copy carries no per-handle state.
// Bin-pair form of the filterbank for the packed (FFMA2) mel stage: the power tile stores bins 2q, 2q+1 of one
// frame side by side, filter m covers pair rows mel_q0(m) .. mel_q0(m) + mel_nq(m) - 1 and its weights are
// stored as (w[2q], w[2q+1]) with zeros outside [kMelLo, kMelHi).
constexpr int kP2Pitch = 66;                       // floats per pair row: 32 columns x 2 bins, + 2 (== 2 mod 32)
constexpr int kP2FirstRow = kMelFirstBin / 2;      // bins below 10 carry no mel weight
constexpr int kP2Rows = kBins / 2 - kP2FirstRow;   // 123
constexpr int kP2RowsAlloc = kP2Rows + 1;          // + the row "bin 256" lands in: a write-only sink that makes every
                                                   // power store unconditional (bins below the first mel bin go there too)
constexpr int mel_q0(int m) { return kMelLo[m] >> 1; }
constexpr int mel_nq(int m) { return ((kMelHi[m] - 1) >> 1) - (kMelLo[m] >> 1) + 1; }
constexpr int mel_qoff(int m) {
  int s = 0;
  for (int i = 0; i < m; ++i) s += mel_nq(i);
  return s;
}
constexpr int kMelPairs = mel_qoff(kNMel);

struct alignas(16) MelDctTables {
  float melw2[2 * kMelPairs + 2];  // pair weights x 2^-20, filter-major (mel_qoff); first: 16-byte aligned for LDCU.128
  float dctp[7][kNMel][2];         // (M[2p][n], M[2p + 1][n]) for the coefficient pair a warp owns, p = 0 .. 6 (M[13] = 0)
  float melw[448];                 // 444 non-zero triangle weights x 2^-20, filter-major (kMelOff)
  float dct[kNCep * kNMel];        // M = lifter[k] * dct2_ortho[k][n] * log10(2)   (input is log2 E)
};
VADB_CONSTANT MelDctTables c_tab;

// FFN weights are per handle (one analyser == one classifier, sklearn_analyser.py:21-35): they
// travel as a __grid_constant__ kernel parameter (constant bank 0: uniform FFMA operands), never
// through device-global state.
struct FfnParams {
  float W1[kNFeat * kH1];        // Keras (in,out) layout: y = x.W + b
  float b1[kH1];
  float W2[kH1 * kH2];
  float b2[kH2];
  float W3[kH2 * kH3];
  float b3[kH3];
  float W4[kH3 * kNCls];
  float b4[kNCls];
  float thresh;                  // decision threshold on p(voiced); <= 0: argmax (vadb200_set_decision_threshold)
};
struct alignas(8) FfnBias {      // what the tensor-core FFN needs besides its weight blob
  float b1[kH1], b2[kH2], b3[kH3], b4[kNCls], thresh;  // thresh: as FfnParams::thresh
  float pre[4];                  // fp16 operand path: power-of-two scale of layer l's input activations (pre[0] == 1)
  float post[4];                 // ... and the exact inverse of (weight scale x activation scale)
  // fp16 path, hidden layers: the next layer's activation scale folded into this layer's epilogue (powers of two,
  // so relu(d post + b) pre' == relu(d (post pre') + b pre') bit for bit): c_l = b_l pre[l+1], postp[l] = post[l] pre[l+1]
  float c1[kH1], c2[kH2], c3[kH3];
  float postp[4];
};
struct FfnNone { int unused; };

struct cf2 { float x, y; };  // layout-compatible with float2 on both sides

// ---- value types: float (one frame per thread) or f2 (two frames per thread, packed) ------------
// sm_100a executes FFMA2 / FADD2 / FMUL2 on register pairs: one issue slot for two lanes of fp32
// work, scalar operands broadcast for free (immediate, uniform register or R.F32).  The FFT code
// below is written once over V; with V = f2 each thread carries the same butterfly for two frames.
#if defined(__CUDACC__)
using f2 = float2;
#else
struct f2 { float x, y; };
#endif
VADB_HD f2 mk2(float a, float b) { f2 r; r.x = a; r.y = b; return r; }
VADB_HD f2 vneg(f2 a) { return mk2(-a.x, -a.y); }
VADB_HD float vneg(float a) { return -a; }
VADB_HD float vadd(float a, float b) { return a + b; }
VADB_HD float vsub(float a, float b) { return a - b; }
VADB_HD float vmul(float a, float b) { return a * b; }
VADB_HD float vmuls(float s, float b) { return s * b; }
VADB_HD float vfma(float a, float b, float c) { return fmaf(a, b, c); }
VADB_HD float vfmas(float s, float b, float c) { return fmaf(s, b, c); }
#if defined(__CUDA_ARCH__)
VADB_HD f2 vadd(f2 a, f2 b) { return __fadd2_rn(a, b); }
VADB_HD f2 vsub(f2 a, f2 b) { return __fadd2_rn(a, vneg(b)); }
VADB_HD f2 vmul(f2 a, f2 b) { return __fmul2_rn(a, b); }
VADB_HD f2 vmuls(float s, f2 b) { return __fmul2_rn(mk2(s, s), b); }
VADB_HD f2 vfma(f2 a, f2 b, f2 c) { return __ffma2_rn(a, b, c); }
VADB_HD f2 vfmas(float s, f2 b, f2 c) { return __ffma2_rn(mk2(s, s), b, c); }
#else
VADB_HD f2 vadd(f2 a, f2 b) { return mk2(a.x + b.x, a.y + b.y); }
VADB_HD f2 vsub(f2 a, f2 b) { return mk2(a.x - b.x, a.y - b.y); }
VADB_HD f2 vmul(f2 a, f2 b) { return mk2(a.x * b.x, a.y * b.y); }
VADB_HD f2 vmuls(float s, f2 b) { return mk2(s * b.x, s * b.y); }
VADB_HD f2 vfma(f2 a, f2 b, f2 c) { return mk2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)); }
VADB_HD f2 vfmas(float s, f2 b, f2 c) { return mk2(fmaf(s, b.x, c.x), fmaf(s, b.y, c.y)); }
#endif
VADB_HD float vzero(float) { return 0.0f; }
VADB_HD f2 vzero(f2) { return mk2(0.0f, 0.0f); }

template <int B, int E, class F>
VADB_HD void static_for(F&& f) {
  if constexpr (B < E) {
    f(std::integral_constant<int, B>{});
    static_for<B + 1, E>(f);
  }
}

// ---- radix-2 butterfly with compile-time twiddle W16^E:  o0 = a + w b,  o1 = a - w b -------
template <int E, class V>
VADB_HD void bfly(V ar, V ai, V br, V bi, V& o0r, V& o0i, V& o1r, V& o1i) {
  constexpr float C1 = 0.92387953251128674f;  // cos(pi/8)
  constexpr float S1 = 0.38268343236508977f;  // sin(pi/8)
  constexpr float R = 0.70710678118654752f;   // sqrt(1/2)
  if constexpr (E == 0) {
    o0r = vadd(ar, br); o0i = vadd(ai, bi); o1r = vsub(ar, br); o1i = vsub(ai, bi);
  } else if constexpr (E == 4) {  // w = -i : w b = (bi, -br)
    o0r = vadd(ar, bi); o0i = vsub(ai, br); o1r = vsub(ar, bi); o1i = vadd(ai, br);
  } else if constexpr (E == 2) {  // w = R(1 - i) : w b = R(br + bi) + i R(bi - br)
    const V s = vadd(br, bi), d = vsub(bi, br);
    o0r = vfmas(R, s, ar); o0i = vfmas(R, d, ai); o1r = vfmas(-R, s, ar); o1i = vfmas(-R, d, ai);
  } else if constexpr (E == 6) {  // w = R(-1 - i) : w b = R(bi - br) - i R(br + bi)
    const V s = vadd(br, bi), d = vsub(bi, br);
    o0r = vfmas(R, d, ar); o0i = vfmas(-R, s, ai); o1r = vfmas(-R, d, ar); o1i = vfmas(R, s, ai);
  } else {  // general: 6 FMA
    constexpr float wr = (E == 1) ? C1 : (E == 3) ? S1 : (E == 5) ? -S1 : -C1;
    constexpr float wi = (E == 1) ? -S1 : (E == 3) ? -C1 : (E == 5) ? -C1 : -S1;
    V xr = vfmas(wr, br, ar); xr = vfmas(-wi, bi, xr);
    V xi = vfmas(wr, bi, ai); xi = vfmas(wi, br, xi);
    o0r = xr; o0i = xi;
    o1r = vfmas(2.0f, ar, vneg(xr)); o1i = vfmas(2.0f, ai, vneg(xi));
  }
}

// 16-point forward DFT (e^{-2 pi i nk/16}), natural order in and out, decimation in time.
// Stage with sub-length m (G = 8/m classes): a = F_m,n[k] at n + 2Gk, b at a + G,
// twiddle W16^(kG), results at n + Gk and n + Gk + 8.  Inputs with index >= NZ are zero.
template <int NZ, class V>
VADB_HD void dft16(V (&xr)[16], V (&xi)[16]) {
  V ar[16], ai[16];
  static_for<0, 8>([&](auto N) {  // m = 1, G = 8
    constexpr int n = N;
    if constexpr (n + 8 < NZ) {
      bfly<0>(xr[n], xi[n], xr[n + 8], xi[n + 8], ar[n], ai[n], ar[n + 8], ai[n + 8]);
    } else {
      ar[n] = xr[n]; ai[n] = xi[n]; ar[n + 8] = xr[n]; ai[n + 8] = xi[n];
    }
  });
  static_for<0, 4>([&](auto N) {  // m = 2, G = 4
    constexpr int n = N;
    static_for<0, 2>([&](auto K) {
      constexpr int k = K, ia = n + 8 * k, ib = ia + 4, o = n + 4 * k;
      bfly<4 * k>(ar[ia], ai[ia], ar[ib], ai[ib], xr[o], xi[o], xr[o + 8], xi[o + 8]);
    });
  });
  static_for<0, 2>([&](auto N) {  // m = 4, G = 2
    constexpr int n = N;
    static_for<0, 4>([&](auto K) {
      constexpr int k = K, ia = n + 4 * k, ib = ia + 2, o = n + 2 * k;
      bfly<2 * k>(xr[ia], xi[ia], xr[ib], xi[ib], ar[o], ai[o], ar[o + 8], ai[o + 8]);
    });
  });
  static_for<0, 8>([&](auto K) {  // m = 8, G = 1
    constexpr int k = K, ia = 2 * k, ib = ia + 1;
    bfly<k>(ar[ia], ai[ia], ar[ib], ai[ib], xr[k], xi[k], xr[k + 8], xi[k + 8]);
  });
}

// ---- pass 1: load, pruned DFT16, inter-pass twiddle -----------------------------------------
// Packed int16 PCM: w32 points at the frame's first sample viewed as 32-bit words (sample
// offset even); thread t takes complex samples t + 16 j (j = 12 only for t < 8: n < 200).
#if defined(__CUDA_ARCH__)
// ALU-pipe conversion: sign-extend (PRMT / SHF) + I2FP.F32.S32 instead of the quarter-rate XU instruction I2F.S16
// (exact either way; -0.8 % on the fused kernel: the XU pipe also serves MUFU and sits behind the shared-memory queue)
VADB_HD float pcm_lo(uint32_t v) {
  int lo;
  asm("prmt.b32 %0, %1, 0, 0x9910;" : "=r"(lo) : "r"(v));
  return __int2float_rn(lo);
}
VADB_HD float pcm_hi(uint32_t v) { return __int2float_rn(static_cast<int>(v) >> 16); }
#else
VADB_HD float pcm_lo(uint32_t v) { return static_cast<float>(static_cast<int16_t>(v & 0xffffu)); }
VADB_HD float pcm_hi(uint32_t v) { return static_cast<float>(static_cast<int16_t>(v >> 16)); }  // I2F.S16 Rx.H1
#endif
VADB_HD void fft_load_pcm(const uint32_t* w32, int t, float (&xr)[16], float (&xi)[16]) {
  static_for<0, 13>([&](auto J) {
    constexpr int j = J;
    uint32_t v = (j < 12 || t < 8) ? w32[t + 16 * j] : 0u;
    xr[j] = pcm_lo(v);
    xi[j] = pcm_hi(v);
  });
  xr[13] = xi[13] = xr[14] = xi[14] = xr[15] = xi[15] = 0.0f;
}
// Two frames per thread: frame A at w32, frame B `delta` words further (same stage buffer).
VADB_HD void fft_load_pcm2(const uint32_t* w32, int delta, int t, f2 (&xr)[16], f2 (&xi)[16]) {
  static_for<0, 13>([&](auto J) {
    constexpr int j = J;
    const bool on = (j < 12 || t < 8);
    const uint32_t va = on ? w32[t + 16 * j] : 0u;
    const uint32_t vb = on ? w32[delta + t + 16 * j] : 0u;
    xr[j] = mk2(pcm_lo(va), pcm_lo(vb));
    xi[j] = mk2(pcm_hi(va), pcm_hi(vb));
  });
  xr[13] = xi[13] = xr[14] = xi[14] = xr[15] = xi[15] = mk2(0.0f, 0.0f);
}

// Explicit float32 frames (the reference's per-frame API takes float frames, vad.py:37).
VADB_HD void fft_load_f32(const float* fr, int frame_len, int t, float (&xr)[16],
                          float (&xi)[16]) {
  static_for<0, 16>([&](auto J) {
    constexpr int j = J;
    const int n = 2 * (t + 16 * j);
    xr[j] = (n < frame_len) ? fr[n] : 0.0f;
    xi[j] = (n + 1 < frame_len) ? fr[n + 1] : 0.0f;
  });
}

// ---- opt-in front end (vadb200_set_frontend): pre-emphasis y[n] = x[n] - a x[n-1], then window weights ----------
// w2[m] = (w[2m], w[2m+1]): a 400-point window (ones when none is set; 256 pairs, entries past 400 are 1).
#if defined(__CUDA_ARCH__)
VADB_HD cf2 win_pair(const cf2* w2, int m) {  // read-only path: every CTA reads the same 2 KB, it stays in L1
  const float2 v = __ldg(reinterpret_cast<const float2*>(w2) + m);
  return cf2{v.x, v.y};
}
#else
VADB_HD cf2 win_pair(const cf2* w2, int m) { return w2[m]; }
#endif
// fft_load_pcm2 with the front end.  Word m - 1 carries x[2m - 1] in its high half: for m = 0, w32[-1] must hold the
// sample before the frame (0 at an utterance start); frame B's word -1 is frame A's data.  The previous word is a
// second shared-memory load per word (same banks pattern as the first: conflict free).
VADB_HD void fft_load_pcm2_fe(const uint32_t* w32, int delta, int t, float a, const cf2* w2, f2 (&xr)[16],
                              f2 (&xi)[16]) {
  static_for<0, 13>([&](auto J) {
    constexpr int j = J;
    const bool on = (j < 12 || t < 8);
    const int m = t + 16 * j;
    const uint32_t va = on ? w32[m] : 0u, pa = on ? w32[m - 1] : 0u;
    const uint32_t vb = on ? w32[delta + m] : 0u, pb = on ? w32[delta + m - 1] : 0u;
    const cf2 w = on ? win_pair(w2, m) : cf2{0.0f, 0.0f};
    const f2 lo = mk2(pcm_lo(va), pcm_lo(vb)), hi = mk2(pcm_hi(va), pcm_hi(vb)), prev = mk2(pcm_hi(pa), pcm_hi(pb));
    xr[j] = vmuls(w.x, vfmas(-a, prev, lo));  // y[2m]     = x[2m]     - a x[2m - 1]
    xi[j] = vmuls(w.y, vfmas(-a, lo, hi));    // y[2m + 1] = x[2m + 1] - a x[2m]
  });
  xr[13] = xi[13] = xr[14] = xi[14] = xr[15] = xi[15] = mk2(0.0f, 0.0f);
}
// fft_load_f32 with the front end; each frame is its own signal (y[0] = x[0]).
VADB_HD void fft_load_f32_fe(const float* fr, int frame_len, int t, float a, const cf2* w2, float (&xr)[16],
                             float (&xi)[16]) {
  static_for<0, 16>([&](auto J) {
    constexpr int j = J;
    const int m = t + 16 * j, n = 2 * m;
    const float x0 = (n < frame_len) ? fr[n] : 0.0f;
    const float x1 = (n + 1 < frame_len) ? fr[n + 1] : 0.0f;
    const float xp = (n > 0 && n < frame_len) ? fr[n - 1] : 0.0f;
    const cf2 w = win_pair(w2, m);
    xr[j] = w.x * fmaf(-a, xp, x0);
    xi[j] = (n + 1 < frame_len) ? w.y * fmaf(-a, x0, x1) : 0.0f;  // zero padding stays zero
  });
}

// tw1: [k1][t] = W256^(t k1).  TW1 is a callable (k1 -> cf2): shared-memory table reads.  The
// twiddle is a per-thread scalar pair; with V = f2 it is broadcast to both frames (R.F32 operand).
template <int NZ, class V, class TW1>
VADB_HD void fft_pass1_tw(V (&xr)[16], V (&xi)[16], TW1&& tw1) {
  dft16<NZ>(xr, xi);
  static_for<1, 16>([&](auto K) {
    constexpr int k1 = K;
    const cf2 w = tw1(K);
    const V r = xr[k1], i = xi[k1];
    xr[k1] = vfmas(w.x, r, vneg(vmuls(w.y, i)));
    xi[k1] = vfmas(w.y, r, vmuls(w.x, i));
  });
}
template <int NZ, class V>
VADB_HD void fft_pass1(V (&xr)[16], V (&xi)[16], const cf2* tw1, int t) {
  fft_pass1_tw<NZ>(xr, xi, [&](auto K) { return tw1[decltype(K)::value * 16 + t]; });
}

// 16x16 transpose buffer of one frame: row n2 = t (pass-1 thread), column k1; row pitch 17
// 64-bit slots (34 words): the 16 threads' 64-bit row stores land on banks 2t, 2t+1 and the 64-bit
// column loads on consecutive words -- both bank-conflict free.  One frame per thread: a slot is
// one complex value (re, im).  Two frames per thread: a slot is one component of both frames
// (A, B), and the real and imaginary planes go through the same buffer one after the other
// (exch_store_plane / exch_load_plane with a warp barrier between), so the scratch does not grow.
constexpr int kExchPitch = 17;
constexpr int kExchFrame = 16 * kExchPitch;  // 64-bit slots per half-warp

VADB_HD void exch_store(cf2* ex, int t, const float (&xr)[16], const float (&xi)[16]) {
  static_for<0, 16>([&](auto K) {
    constexpr int k1 = K;
    ex[t * kExchPitch + k1] = cf2{xr[k1], xi[k1]};
  });
}
VADB_HD void exch_load(const cf2* ex, int k1, float (&xr)[16], float (&xi)[16]) {
  static_for<0, 16>([&](auto N) {
    constexpr int n2 = N;
    const cf2 v = ex[n2 * kExchPitch + k1];
    xr[n2] = v.x; xi[n2] = v.y;
  });
}
VADB_HD void exch_store_plane(f2* ex, int t, const f2 (&x)[16]) {
  static_for<0, 16>([&](auto K) { ex[t * kExchPitch + decltype(K)::value] = x[decltype(K)::value]; });
}
VADB_HD void exch_load_plane(const f2* ex, int k1, f2 (&x)[16]) {
  static_for<0, 16>([&](auto N) { x[decltype(N)::value] = ex[decltype(N)::value * kExchPitch + k1]; });
}

// ---- real-FFT split of one bin pair (k, 256-k); returns |2 X[k]|^2 and |2 X[256-k]|^2 -------
template <class V>
VADB_HD void split_pair(V ar, V ai, V br, V bi, float wr, float wi, V& plo, V& phi) {
  const V er = vadd(ar, br), ei = vsub(ai, bi);    // E = a + conj(b)
  const V qr = vadd(ai, bi), qi = vsub(br, ar);    // O = -i (a - conj(b))
  V xr = vfmas(wr, qr, er); xr = vfmas(-wi, qi, xr);   // 2 X[k] = E + w O
  V xi = vfmas(wr, qi, ei); xi = vfmas(wi, qr, xi);
  const V yr = vfmas(2.0f, er, vneg(xr)), yi = vfmas(2.0f, ei, vneg(xi));  // 2 conj X[256-k] = E - w O
  plo = vfma(xr, xr, vmul(xi, xi));
  phi = vfma(yr, yr, vmul(yi, yi));
}

// After pass 2 thread k1 holds Z[k1 + 16 k2] in (xr[k2], xi[k2]).  It finishes the 8 pairs
// (k, 256-k), k = k1 + 16 k2, k2 < 8; the mirror element is Z[(16-k1) + 16 (15-k2)] on the
// partner thread.  Thread 0 pairs with itself at index 16 - k2, so it rotates its send
// registers by one; it also owns the self-paired bin 128 (|X|^2 = |Z|^2).
// XCH(mine, j, is_imag, partner) returns the partner's send register j.
// store(bin, value) receives raw power |2X|^2 for bins 0..255.
#if defined(__CUDACC__)
#pragma nv_exec_check_disable
#endif
// STORE::kHasSink: the store redirects bins it does not keep (and bin 256) to a sink row, so every store below is
// unconditional -- no divergent branches around the first pair, the (0, 256) pair and thread 0's bin 128.
template <class S, class = void> struct store_has_sink { static constexpr bool value = false; };
template <class S> struct store_has_sink<S, std::enable_if_t<S::kHasSink>> { static constexpr bool value = true; };

template <class V, class TW2, class XCH, class STORE>
VADB_HD void fft_split_store_tw(const V (&xr)[16], const V (&xi)[16], int k1, TW2&& tw2,
                                XCH&& xch, STORE&& store) {
  constexpr bool kSink = store_has_sink<std::remove_cv_t<std::remove_reference_t<STORE>>>::value;
  V sr[16], si[16];
  static_for<8, 16>([&](auto J) {
    constexpr int j = J;
    sr[j] = (k1 == 0) ? xr[(j + 1) & 15] : xr[j];
    si[j] = (k1 == 0) ? xi[(j + 1) & 15] : xi[j];
  });
  const int partner = (16 - k1) & 15;
  static_for<0, 8>([&](auto K) {
    constexpr int k2 = K;
    const V br = xch(sr[15 - k2], 15 - k2, false, partner);
    const V bi = xch(si[15 - k2], 15 - k2, true, partner);
    const cf2 w = tw2(K);  // W512^(k1 + 16 k2)
    V plo, phi;
    split_pair(xr[k2], xi[k2], br, bi, w.x, w.y, plo, phi);
    if constexpr (kSink) {   // addresses are affine in k2: the store keeps per-thread base pointers
      store.lo(K, plo);
      store.hi(K, phi);      // thread 0's (0, 256) pair: bin 256 is the sink
    } else {
      const int lo = k1 + 16 * k2;
      store(lo, plo);
      if (k2 != 0 || k1 != 0) store(256 - lo, phi);
    }
  });
  if constexpr (kSink) {
    store.mid(vmuls(4.0f, vfma(xr[8], xr[8], vmul(xi[8], xi[8]))));   // bin 128 on thread 0, sink elsewhere
  } else {
    if (k1 == 0) store(128, vmuls(4.0f, vfma(xr[8], xr[8], vmul(xi[8], xi[8]))));
  }
}
#if defined(__CUDACC__)
#pragma nv_exec_check_disable
#endif
template <class V, class XCH, class STORE>
VADB_HD void fft_split_store(const V (&xr)[16], const V (&xi)[16], int k1, const cf2* tw2,
                             XCH&& xch, STORE&& store) {
  fft_split_store_tw(xr, xi, k1, [&](auto K) { return tw2[decltype(K)::value * 16 + k1]; }, xch, store);
}

// ---- mel + log: lane = frame; P points at column `lane` of the [256][pitch] power tile -------
VADB_HD float log2_energy(float e) {
  // mfcc.py:74: exact zeros -> float64 eps = 2^-52 (exactly representable in fp32)
  e = (e == 0.0f) ? 2.220446049250313e-16f : e;
#if defined(__CUDA_ARCH__)
  // MUFU.LG2 (CUDA C++ Programming Guide, intrinsic functions): absolute error <= 2^-22 for e in [0.5, 2], else
  // <= 2 ulp of the result; tests/_mfcc_bound.py holds the MFCC rows to exactly this
  return __log2f(e);
#else
  return log2f(e);
#endif
}

template <int G, int PITCH, int OPITCH>
VADB_HD void mel_group(const float* P, float* logE) {
  static_for<0, kMelGroupCount[G]>([&](auto J) {
    constexpr int m = kMelGroupFilter[G][J];
    constexpr int lo = kMelLo[m], hi = kMelHi[m], off = kMelOff[m];
    float e0 = 0.0f, e1 = 0.0f, e2 = 0.0f, e3 = 0.0f;  // four chains: dependent-FFMA latency / 4
    static_for<lo, hi>([&](auto K) {
      constexpr int k = K;
      constexpr int c = (k - lo) & 3;
      const float pw = P[k * PITCH];
      const float w = c_tab.melw[off + k - lo];
      if constexpr (c == 0) e0 = fmaf(pw, w, e0);
      else if constexpr (c == 1) e1 = fmaf(pw, w, e1);
      else if constexpr (c == 2) e2 = fmaf(pw, w, e2);
      else e3 = fmaf(pw, w, e3);
    });
    e0 = (e0 + e2) + (e1 + e3);
    e1 = 0.0f;
    logE[m * OPITCH] = log2_energy(e0 + e1);
  });
}

template <int PITCH, int OPITCH>
VADB_HD void mel_group_dispatch(int g, const float* P, float* logE) {
  switch (g) {
    case 0: mel_group<0, PITCH, OPITCH>(P, logE); break;
    case 1: mel_group<1, PITCH, OPITCH>(P, logE); break;
    case 2: mel_group<2, PITCH, OPITCH>(P, logE); break;
    case 3: mel_group<3, PITCH, OPITCH>(P, logE); break;
    case 4: mel_group<4, PITCH, OPITCH>(P, logE); break;
    case 5: mel_group<5, PITCH, OPITCH>(P, logE); break;
    case 6: mel_group<6, PITCH, OPITCH>(P, logE); break;
    default: mel_group<7, PITCH, OPITCH>(P, logE); break;
  }
}

// Load-sharing packed mel: P2 points at this lane's column of the pair tile (row r = pair row - kP2FirstRow at
// P2 + r * PITCH2, two floats = bins 2q, 2q+1).  Warp g owns the run of consecutive filters kMelRunFirst[g] ..
// kMelRunLast[g] and walks the pair rows they cover once -- every power pair is loaded a single time (LDS.64) and feeds each filter whose triangle
// contains it (neighbouring triangles overlap by half: two FFMA2 per load in the interior).  Two accumulator chains per
// filter; with two or three filters live per row that is four to six independent FFMA2 chains.
template <int G, int PITCH2, int OPITCH>
VADB_HD void mel2_run(const float* P2, float* logE) {
  constexpr int m0 = kMelRunFirst[G], m1 = kMelRunLast[G], nf = m1 - m0 + 1;
  if constexpr (nf > 0) {
  constexpr int qa = mel_q0(m0), qb = mel_q0(m1) + mel_nq(m1);   // pair rows [qa, qb)
  f2 acc[nf][2];
  static_for<0, nf>([&](auto F) { acc[F][0] = mk2(0.0f, 0.0f); acc[F][1] = mk2(0.0f, 0.0f); });
  static_for<qa, qb>([&](auto Q) {
    constexpr int q = Q;
    const float* pp = P2 + (q - kP2FirstRow) * PITCH2;
    const f2 pv = mk2(pp[0], pp[1]);
    static_for<0, nf>([&](auto F) {
      constexpr int m = m0 + F;
      if constexpr (q >= mel_q0(m) && q < mel_q0(m) + mel_nq(m)) {
        constexpr int i = q - mel_q0(m), off = mel_qoff(m);
        const f2 wv = mk2(c_tab.melw2[2 * (off + i)], c_tab.melw2[2 * (off + i) + 1]);
        acc[F][i & 1] = vfma(pv, wv, acc[F][i & 1]);
      }
    });
    // a filter whose last row this was is finished: log and store it while the others continue
    static_for<0, nf>([&](auto F) {
      constexpr int m = m0 + F;
      if constexpr (q == mel_q0(m) + mel_nq(m) - 1) {
        const f2 sacc = vadd(acc[F][0], acc[F][1]);
        logE[m * OPITCH] = log2_energy(sacc.x + sacc.y);
      }
    });
  });
  }  // warps without filters do nothing
}
template <int PITCH2, int OPITCH>
VADB_HD void mel2_run_dispatch(int g, const float* P2, float* logE) {
  switch (g) {
    case 0: mel2_run<0, PITCH2, OPITCH>(P2, logE); break;
    case 1: mel2_run<1, PITCH2, OPITCH>(P2, logE); break;
    case 2: mel2_run<2, PITCH2, OPITCH>(P2, logE); break;
    case 3: mel2_run<3, PITCH2, OPITCH>(P2, logE); break;
    case 4: mel2_run<4, PITCH2, OPITCH>(P2, logE); break;
    case 5: mel2_run<5, PITCH2, OPITCH>(P2, logE); break;
    case 6: mel2_run<6, PITCH2, OPITCH>(P2, logE); break;
    default: mel2_run<7, PITCH2, OPITCH>(P2, logE); break;
  }
}
// Who owns which column of the 32-frame step.  Half-warp h of warp w carries frame slots 4w + h and 4w + h + 2 (PCM of
// neighbouring slots is 80 words apart, so the two half-warps read different banks) and stores them in adjacent
// columns c, c + 1 with c = 2 (w & 3) + 8 h + 16 (w >> 2): the second half-warp's columns are 8 further, i.e. 16
// banks, which makes the 32-lane power stores conflict free.
VADB_HD int col_of_halfwarp(int w, int h) { return 2 * (w & 3) + 8 * h + 16 * (w >> 2); }
VADB_HD int slot_of_col(int c) {
  const int q = c >> 1, w = (q & 3) + 4 * (q >> 3);
  return 4 * w + ((q >> 2) & 1) + 2 * (c & 1);
}
// offset (floats) of power bin `bin` of column `col` in the pair tile
VADB_HD int p2_index(int bin, int col) { return ((bin >> 1) - kP2FirstRow) * kP2Pitch + 2 * col + (bin & 1); }

// DCT-II(ortho)[:13] x lifter x log10(2) of the 26 log2-energies of one frame (column).
template <int PITCH>
VADB_HD float dct_coef(const float* logE, int c) {
  float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;  // four chains instead of one 26-long one
#pragma unroll
  for (int n = 0; n < 24; n += 4) {
    a0 = fmaf(logE[(n + 0) * PITCH], c_tab.dct[c * kNMel + n + 0], a0);
    a1 = fmaf(logE[(n + 1) * PITCH], c_tab.dct[c * kNMel + n + 1], a1);
    a2 = fmaf(logE[(n + 2) * PITCH], c_tab.dct[c * kNMel + n + 2], a2);
    a3 = fmaf(logE[(n + 3) * PITCH], c_tab.dct[c * kNMel + n + 3], a3);
  }
  a0 = fmaf(logE[24 * PITCH], c_tab.dct[c * kNMel + 24], a0);
  a1 = fmaf(logE[25 * PITCH], c_tab.dct[c * kNMel + 25], a1);
  return (a0 + a2) + (a1 + a3);
}

// Coefficients 2p and 2p + 1 of the same frame at once (p = 0 .. 6; coefficient 13 is a zero row): one FFMA2 per
// log-energy on the coefficient pair, the log-energy broadcast to both halves.  Per coefficient the chains are those
// of dct_coef (bit-identical).  The pair is what one 64-bit slot of the fused kernels' MFCC ring holds.
template <int PITCH>
VADB_HD void dct_coef2(const float* logE, int p, float& ra, float& rb) {
  f2 a0 = mk2(0.0f, 0.0f), a1 = a0, a2 = a0, a3 = a0;
  const float (*w)[2] = c_tab.dctp[p];
#pragma unroll
  for (int n = 0; n < 24; n += 4) {
    a0 = vfmas(logE[(n + 0) * PITCH], mk2(w[n + 0][0], w[n + 0][1]), a0);
    a1 = vfmas(logE[(n + 1) * PITCH], mk2(w[n + 1][0], w[n + 1][1]), a1);
    a2 = vfmas(logE[(n + 2) * PITCH], mk2(w[n + 2][0], w[n + 2][1]), a2);
    a3 = vfmas(logE[(n + 3) * PITCH], mk2(w[n + 3][0], w[n + 3][1]), a3);
  }
  a0 = vfmas(logE[24 * PITCH], mk2(w[24][0], w[24][1]), a0);
  a1 = vfmas(logE[25 * PITCH], mk2(w[25][0], w[25][1]), a1);
  const f2 r = vadd(vadd(a0, a2), vadd(a1, a3));
  ra = r.x;
  rb = r.y;
}

// Two coefficient pairs (p, p + 1) of the same frame from one pass over the 26 log-energies: the loads are shared,
// the eight FFMA2 chains are those of two dct_coef2 calls (bit-identical results).
template <int PITCH>
VADB_HD void dct_coef4(const float* logE, int p, float& ra, float& rb, float& rc, float& rd) {
  f2 a0 = mk2(0.0f, 0.0f), a1 = a0, a2 = a0, a3 = a0, b0 = a0, b1 = a0, b2 = a0, b3 = a0;
  const float (*w)[2] = c_tab.dctp[p];
  const float (*v)[2] = c_tab.dctp[p + 1];
#pragma unroll
  for (int n = 0; n < 24; n += 4) {
    const float e0 = logE[(n + 0) * PITCH], e1 = logE[(n + 1) * PITCH], e2 = logE[(n + 2) * PITCH],
                e3 = logE[(n + 3) * PITCH];
    a0 = vfmas(e0, mk2(w[n + 0][0], w[n + 0][1]), a0);
    b0 = vfmas(e0, mk2(v[n + 0][0], v[n + 0][1]), b0);
    a1 = vfmas(e1, mk2(w[n + 1][0], w[n + 1][1]), a1);
    b1 = vfmas(e1, mk2(v[n + 1][0], v[n + 1][1]), b1);
    a2 = vfmas(e2, mk2(w[n + 2][0], w[n + 2][1]), a2);
    b2 = vfmas(e2, mk2(v[n + 2][0], v[n + 2][1]), b2);
    a3 = vfmas(e3, mk2(w[n + 3][0], w[n + 3][1]), a3);
    b3 = vfmas(e3, mk2(v[n + 3][0], v[n + 3][1]), b3);
  }
  const float e24 = logE[24 * PITCH], e25 = logE[25 * PITCH];
  a0 = vfmas(e24, mk2(w[24][0], w[24][1]), a0);
  b0 = vfmas(e24, mk2(v[24][0], v[24][1]), b0);
  a1 = vfmas(e25, mk2(w[25][0], w[25][1]), a1);
  b1 = vfmas(e25, mk2(v[25][0], v[25][1]), b1);
  const f2 r = vadd(vadd(a0, a2), vadd(a1, a3)), q = vadd(vadd(b0, b2), vadd(b1, b3));
  ra = r.x; rb = r.y; rc = q.x; rd = q.y;
}

// A product rounded on its own: nvcc contracts a plain product into the add or subtract that consumes it (FFMA),
// which the packed path (__fmul2_rn) never does.  The window features' mean and z use it, here and in the stream
// kernel, so fp32, tc and tc16 classify the same features.
VADB_HD float mul_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}

VADB_HD float vadb_rsqrt(float v) {
#if defined(__CUDA_ARCH__)
  return rsqrtf(v);  // MUFU.RSQ, <= 2 ulp
#else
  return 1.0f / sqrtf(v);
#endif
}

// ---- 5-frame window features ------------------------------------------------------------------
// r[d][k] = MFCC k of frame t-2+d.  mode 0: analyser (sklearn_analyser.py:52-69,103-107);
// mode 1: dataset (file_processing.py:51-66).  Returns false when a feature is non-finite
// (sigma5 == 0: the reference yields nan -> numpy argmax 0 -> non-speech).
VADB_HD bool window_features(const float (&r)[5][kNCep], int mode, float (&x)[kNFeat]) {
  bool ok = true;
#pragma unroll
  for (int k = 0; k < kNCep; ++k) {
    const float c0 = r[0][k], c1 = r[1][k], c2 = r[2][k], c3 = r[3][k], c4 = r[4][k];
    float z = c2;
    if (mode == 0) {
      // mul_rn: rounded like window_features_pairs' FMUL2, so every classifier path sees the same features
      const float mu = mul_rn((((c0 + c1) + c2) + c3) + c4, 0.2f);
      const float d0 = c0 - mu, d1 = c1 - mu, d2 = c2 - mu, d3 = c3 - mu, d4 = c4 - mu;
      const float var = fmaf(d4, d4, fmaf(d3, d3, fmaf(d2, d2, fmaf(d1, d1, d0 * d0)))) * 0.2f;
      // exact-arithmetic semantics of np.std == 0: all five equal -> 0/0 = nan
      const bool alleq = (c0 == c1) && (c1 == c2) && (c2 == c3) && (c3 == c4);
      z = alleq ? NAN : mul_rn(d2, vadb_rsqrt(var));
      ok = ok && (fabsf(z) <= 3.0e38f);  // false for nan and inf
    }
    x[k] = z;
    x[kNCep + k] = c3 - c1;
    x[2 * kNCep + k] = (c4 - z) - (z - c0);
  }
  return ok;
}

// ---- MFCC ring of the fused kernels: coefficient pairs side by side --------------------------------------------------
// Row q holds coefficients 2q, 2q+1 of every slot as one 64-bit element, so the window features of a coefficient pair
// are built with packed (FADD2 / FFMA2 / FMUL2) arithmetic from five LDS.64.  Element 1 of row 6 is never written.
constexpr int kRingRows = (kNCep + 1) / 2;  // 7
VADB_HD constexpr int ring_pitch(int ring) { return 2 * ring + 2; }   // floats per row
VADB_HD constexpr int ring_idx(int k, int slot, int ring) { return (k >> 1) * ring_pitch(ring) + 2 * slot + (k & 1); }

VADB_HD uint32_t fbits(float x) {
#if defined(__CUDA_ARCH__)
  return __float_as_uint(x);
#else
  uint32_t u;
  __builtin_memcpy(&u, &x, 4);
  return u;
#endif
}
// Window features of the coefficient pairs [Q0, Q1), centre frame c, in the layer-1 column order of the
// tensor-core FFN (ffn_tc.cuh tc_feat_col): out[6 j + 2 g + e] = feature g (0 z, 1 d1, 2 d2) of coefficient
// 2 (Q0 + j) + e.  Per coefficient the arithmetic is that of window_features (packed ops round like scalar ones);
// "all five equal" is tested on the bit patterns (+-0 mixes and NaNs end in NaN either way: var = 0 -> 0 x inf).
template <int Q0, int Q1, int RING, int NOUT>
VADB_HD bool window_features_pairs(const float* ring2, int c, int mode, float (&out)[NOUT]) {
  static_assert(6 * (Q1 - Q0) <= NOUT, "output too small");
  constexpr int PITCH = ring_pitch(RING);
  bool ok = true;
  const int i0 = 2 * ((c - 2) % RING), i1 = 2 * ((c - 1) % RING), i2 = 2 * (c % RING), i3 = 2 * ((c + 1) % RING),
            i4 = 2 * ((c + 2) % RING);
#pragma unroll
  for (int q = Q0; q < Q1; ++q) {
    const float* row = ring2 + q * PITCH;
    f2 c0 = mk2(row[i0], row[i0 + 1]), c1 = mk2(row[i1], row[i1 + 1]), c2 = mk2(row[i2], row[i2 + 1]),
       c3 = mk2(row[i3], row[i3 + 1]), c4 = mk2(row[i4], row[i4 + 1]);
    const bool pad = 2 * q + 1 >= kNCep;  // compile-time after unrolling: element 1 is not a coefficient
    if (pad) { c0.y = 0.0f; c1.y = 1.0f; c2.y = 2.0f; c3.y = 3.0f; c4.y = 4.0f; }
    f2 z = c2;
    if (mode == 0) {
      const f2 mu = vmuls(0.2f, vadd(vadd(vadd(vadd(c0, c1), c2), c3), c4));
      const f2 d0 = vsub(c0, mu), d1 = vsub(c1, mu), d2 = vsub(c2, mu), d3 = vsub(c3, mu), d4 = vsub(c4, mu);
      const f2 var = vmuls(0.2f, vfma(d4, d4, vfma(d3, d3, vfma(d2, d2, vfma(d1, d1, vmul(d0, d0))))));
      const bool eqx = ((fbits(c0.x) ^ fbits(c1.x)) | (fbits(c1.x) ^ fbits(c2.x)) | (fbits(c2.x) ^ fbits(c3.x)) |
                        (fbits(c3.x) ^ fbits(c4.x))) == 0u;
      const bool eqy = ((fbits(c0.y) ^ fbits(c1.y)) | (fbits(c1.y) ^ fbits(c2.y)) | (fbits(c2.y) ^ fbits(c3.y)) |
                        (fbits(c3.y) ^ fbits(c4.y))) == 0u;
      z = vmul(d2, mk2(vadb_rsqrt(var.x), vadb_rsqrt(var.y)));
      if (eqx) z.x = NAN;
      if (eqy) z.y = NAN;
      ok = ok && (fabsf(z.x) <= 3.0e38f) && (fabsf(z.y) <= 3.0e38f);
    }
    const f2 e1 = vsub(c3, c1);
    const f2 e2 = vsub(vsub(c4, z), vsub(z, c0));
    float* o = out + 6 * (q - Q0);
    o[0] = z.x;  o[1] = pad ? 0.0f : z.y;
    o[2] = e1.x; o[3] = pad ? 0.0f : e1.y;
    o[4] = e2.x; o[5] = pad ? 0.0f : e2.y;
  }
#pragma unroll
  for (int i = 6 * (Q1 - Q0); i < NOUT; ++i) out[i] = 0.0f;
  return ok;
}

// ---- FFN forward, one frame per thread, weights as uniform constant operands (w = kernel parameter) -------------------
VADB_HD void ffn_forward(const FfnParams& w, const float (&x)[kNFeat], float (&logit)[kNCls]) {
  float h2[kH2];
#pragma unroll
  for (int o = 0; o < kH2; ++o) h2[o] = w.b2[o];
  // Rolled on purpose: the fully unrolled FFN (134 KB of SASS) thrashed the instruction cache
  // (ncu: 33 % stall_no_inst in this phase); one 8-neuron body is ~12 KB.
#pragma unroll 1
  for (int c = 0; c < kH1 / 8; ++c) {  // 8 layer-1 neurons at a time, streamed into layer 2
    float h1[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) h1[j] = w.b1[8 * c + j];
#pragma unroll
    for (int i = 0; i < kNFeat; ++i) {
#pragma unroll
      for (int j = 0; j < 8; ++j) h1[j] = fmaf(x[i], w.W1[i * kH1 + 8 * c + j], h1[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float a = fmaxf(h1[j], 0.0f);  // the duplicate ReLU (ffn_trainer.py:110) is idempotent
#pragma unroll
      for (int o = 0; o < kH2; ++o) h2[o] = fmaf(a, w.W2[(8 * c + j) * kH2 + o], h2[o]);
    }
  }
  float h3[kH3];
#pragma unroll
  for (int o = 0; o < kH3; ++o) h3[o] = w.b3[o];
#pragma unroll
  for (int i = 0; i < kH2; ++i) {
    const float a = fmaxf(h2[i], 0.0f);
#pragma unroll
    for (int o = 0; o < kH3; ++o) h3[o] = fmaf(a, w.W3[i * kH3 + o], h3[o]);
  }
#pragma unroll
  for (int o = 0; o < kNCls; ++o) logit[o] = w.b4[o];
#pragma unroll
  for (int i = 0; i < kH3; ++i) {
    const float a = fmaxf(h3[i], 0.0f);
#pragma unroll
    for (int o = 0; o < kNCls; ++o) logit[o] = fmaf(a, w.W4[i * kNCls + o], logit[o]);
  }
}

// speech <=> argmax == VOICED(1) (sklearn_analyser.py:76, config.py:45-47); numpy argmax
// takes the first maximum, so class 1 must be strictly greater than class 0 and >= class 2.
VADB_HD uint8_t decide(const float (&logit)[kNCls]) {
  return (logit[1] > logit[0] && logit[1] >= logit[2]) ? 1 : 0;
}
// Opt-in operating point: speech <=> softmax(logit)[1] >= th.  th <= 0 keeps the argmax rule.
VADB_HD uint8_t decide(const float (&logit)[kNCls], float th) {
  if (!(th > 0.0f)) return decide(logit);
  const float s = 1.0f + expf(logit[0] - logit[1]) + expf(logit[2] - logit[1]);  // 1 / p(voiced)
  return (1.0f / s >= th) ? 1 : 0;
}

}  // namespace vadb
