// vad_resample.cuh -- audio of any common WAV sample format, channel count and sample rate -> 16 kHz int16 PCM
// (DESIGN.md section 5.8).
//
// decode_pcm_kernel: interleaved frames of C channels in one of six sample formats (little- or big-endian) -> float32
//   in int16 units, the mean of the channels, gathered segment by segment like ingest_kernel.
// resample_kernel<In>: a ragged packed batch at rate r -> 16 kHz int16, y = scipy.signal.resample_poly(x, up, down)
//   rounded half-to-even and saturated.  Output-stationary: one CTA owns a tile of T = 2H consecutive outputs of one
//   utterance, stages the tile's input window and the polyphase taps in shared memory, and each thread runs the tap
//   loop for the output pair (m, m + H) -- the same polyphase row, since H is a multiple of `up` -- as packed FFMA2.
#pragma once

#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <numeric>
#include <vector>

namespace vadb {

// ---- formats (VADB200_PCM_*) ---------------------------------------------------------------------------------
enum PcmFormat { kPcmS16 = 0, kPcmU8 = 1, kPcmS24 = 2, kPcmS32 = 3, kPcmF32 = 4, kPcmF64 = 5 };
constexpr int kPcmBytes[6] = {2, 1, 3, 4, 4, 8};
template <int FMT>
constexpr int kPcmSize = FMT == kPcmU8 ? 1 : FMT == kPcmS16 ? 2 : FMT == kPcmS24 ? 3 : FMT == kPcmF64 ? 8 : 4;
constexpr int kMaxChannels = 32;

// ---- the resampling filter (host) ------------------------------------------------------------------------------
constexpr int kOutRate = 16000;
constexpr int kMaxPhases = 1024;        // max(up, down) <= 1024: at most 20 481 taps
constexpr int kResampleThreads = 256;

struct ResampleDesign {
  int up = 0, down = 0, half = 0, L = 0;   // L = 2 half + 1 taps (identity: half = 0, one tap of 1)
  int K = 0, Ks = 0;                       // taps per polyphase row; row stride in floats (odd: fewer bank conflicts)
  int q = 0, H = 0, T = 0;                 // H = q up outputs per half tile, T = 2 H per tile
  int win = 0;                             // float2 entries of the staged input window
  size_t smem = 0;                         // dynamic shared memory per CTA
};

inline bool resample_ratio(long long rate, int* up, int* down) {
  if (rate < 4000 || rate > 384000) return false;
  const long long g = std::gcd(rate, static_cast<long long>(kOutRate));
  *up = static_cast<int>(kOutRate / g);
  *down = static_cast<int>(rate / g);
  return std::max(*up, *down) <= kMaxPhases;
}

// ceil(n up / down): the length scipy.signal.resample_poly returns
inline long long resampled_length(long long n, int up, int down) { return (n * up + down - 1) / down; }

// Zeroth-order modified Bessel function of the first kind (power series; x <= 5 here, so 30 terms reach 1e-17).
inline double bessel_i0(double x) {
  double term = 1.0, sum = 1.0;
  const double q = 0.25 * x * x;
  for (int k = 1; k < 60; ++k) {
    term *= q / (static_cast<double>(k) * k);
    sum += term;
    if (term < 1e-18 * sum) break;
  }
  return sum;
}

// scipy.signal.firwin(L, 1 / max(up, down), window=('kaiser', 5.0)) * up, in float64 (scale=True: unit DC gain
// before the factor up).  The identity (up == down == 1) is the single tap 1.
inline std::vector<double> resample_taps(int up, int down) {
  if (up == 1 && down == 1) return std::vector<double>(1, 1.0);
  const int mx = std::max(up, down);
  const int half = 10 * mx, L = 2 * half + 1;
  const double fc = 1.0 / mx, alpha = 0.5 * (L - 1), beta = 5.0, i0b = bessel_i0(beta);
  const double pi = 3.14159265358979323846;
  std::vector<double> h(L);
  double s = 0.0;
  for (int n = 0; n < L; ++n) {
    const double m = n - alpha;
    const double y = pi * (m == 0.0 ? 1e-20 : fc * m);   // np.sinc
    const double sinc = std::sin(y) / y;
    const double r = (n - alpha) / alpha;
    const double w = bessel_i0(beta * std::sqrt(std::max(0.0, 1.0 - r * r))) / i0b;
    h[n] = fc * sinc * w;
    s += h[n];
  }
  for (int n = 0; n < L; ++n) h[n] = h[n] / s * up;
  return h;
}

inline ResampleDesign resample_design(int up, int down) {
  ResampleDesign d;
  d.up = up; d.down = down;
  d.half = (up == 1 && down == 1) ? 0 : 10 * std::max(up, down);
  d.L = 2 * d.half + 1;
  d.K = (d.L + up - 1) / up;
  d.Ks = d.K | 1;
  // about 1024 output pairs per CTA (4 per thread), the input window at most 6144 + K pairs
  d.q = std::max(1, std::min((1024 + up - 1) / up, 6144 / down));
  d.H = d.q * up;
  d.T = 2 * d.H;
  d.win = (d.q * down + d.K + 2) & ~1;   // even: the int16 staging after it stays 16-byte aligned
  const size_t taps = (static_cast<size_t>(up) * d.Ks + 3) / 4 * 4;
  d.smem = taps * sizeof(float) + static_cast<size_t>(d.win) * sizeof(float2) + (static_cast<size_t>(d.T) + 8) * 2;
  return d;
}

// Polyphase order: row p holds h[p], h[p + up], h[p + 2 up], ... (zeros past L), rows Ks floats apart.  Output m
// with t = m down + half uses row t mod up against x[t div up - i], i = 0 .. K - 1.
inline std::vector<float> polyphase_taps(const ResampleDesign& d, const std::vector<double>& h) {
  std::vector<float> t(static_cast<size_t>(d.up) * d.Ks, 0.0f);
  for (int p = 0; p < d.up; ++p)
    for (int i = 0; i < d.K; ++i) {
      const long long j = p + static_cast<long long>(i) * d.up;
      if (j < d.L) t[static_cast<size_t>(p) * d.Ks + i] = static_cast<float>(h[j]);
    }
  return t;
}

// One utterance of a resample call: where its input and output start, and its first tile in the launch.
struct ResampleUtt {
  long long in_off, in_len, out_off, tile_begin;
};
// The work list reaches the device inside kernel parameters (no host copy, so a call stays capturable in a graph):
// fill kernels write it into the caller's workspace, kResampleFill utterances per launch.
constexpr int kResampleFill = 960;
struct ResampleFill {
  ResampleUtt u[kResampleFill];
};
static_assert(sizeof(ResampleFill) + 64 < 32764, "kernel parameters are at most 32764 bytes");

struct ResampleParams {
  const void* in;
  int16_t* out;
  const ResampleUtt* utts;
  int n_utt;
  const float* taps;   // [up][Ks]
  int up, down, half, K, Ks, q, H, win;
  int taps_floats;     // up Ks rounded up to 4
};

// Launchers (vad_resample.cu, a translation unit of its own: compiling these kernels next to the fused kernels
// perturbs NVVM's optimisation of the fused kernels, whose SASS must not move).  They only enqueue.
cudaError_t resample_allow_smem(int bytes);
void enqueue_decode_pcm(int fmt, dim3 grid, cudaStream_t st, const uint8_t* raw, int channels, int be,
                        const long long* src, const long long* dst_off, const long long* len, float* dst);
// fills utts[0, n) from `list` (host), then runs the T-output tiles 0 .. tiles - 1
void enqueue_resample(bool s16, const ResampleParams& a, const ResampleUtt* list, long long n, long long tiles,
                      size_t smem, cudaStream_t st);

// ---- the resampling ragged bank (vad_stream_resample.cu, index math in vad_stream_resample.h) -------------------
// What the plan step decides for one stream and feed.
struct SrsFeed {
  long long n0;    // source samples taken before this feed
  long long src;   // the packet's first sample in the caller's samples
  long long out;   // its first new 16 kHz sample in the bank's packed buffer
  int c;           // packet length (0 for a bad one)
  int outs;        // 16 kHz samples it adds
  int rd;          // history buffer holding x[n0 - K + 1 .. n0 - 1]
  int pad;
};
struct StreamResampleParams {
  int n, cap, cap16;
  int up, down, half, K, Ks;
  int hs;                    // history slots per stream: K - 1
  const float* taps;         // [up][Ks] polyphase rows (polyphase_taps)
  long long* n_in;           // [n] source samples taken since the last reset or end
  int* cur;                  // [n] the history buffer the next feed reads
  int16_t* hist;             // [2][n][hs]
  SrsFeed* feed;             // [n]
  int* tile_off;             // [n + 1] first tile of each stream; [n] the feed's tiles
  long long* off16;          // [n + 1] packed 16 kHz offsets (a bad stream: cap16 + 1 samples, never read)
  int16_t* pcm16;            // [n (cap16 + 1)] the feed's 16 kHz samples
  const int16_t* samples;    // the caller's source packets (may be pinned host memory)
  const long long* offsets;  // [n + 1]
};
// Plan (one CTA) then resample (`grid` CTAs looping over the feed's tiles): two launches.
void enqueue_stream_resample(const StreamResampleParams& p, int grid, cudaStream_t st);
// Zero n_in and both histories of the streams with end[i] != 0: one launch.
void enqueue_stream_resample_end(const StreamResampleParams& p, const uint8_t* end, cudaStream_t st);

#if defined(VADB_RESAMPLE_KERNELS)
__global__ void __launch_bounds__(256) resample_fill_kernel(ResampleUtt* dst, int n, const __grid_constant__ ResampleFill f) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = f.u[i];
}

template <class In>
__device__ __forceinline__ float resample_load(const In* p, long long i) {
  if constexpr (sizeof(In) == 2) return static_cast<float>(static_cast<int>(p[i]));
  else return p[i];
}

template <class In>
__global__ void __launch_bounds__(kResampleThreads) resample_kernel(const ResampleParams a) {
  extern __shared__ float4 smem_f4[];
  float* s_taps = reinterpret_cast<float*>(smem_f4);
  float2* s_z = reinterpret_cast<float2*>(s_taps + a.taps_floats);
  int16_t* s_out = reinterpret_cast<int16_t*>(s_z + a.win);
  const int tid = threadIdx.x;
  // utterance of this tile: the last one whose first tile is <= blockIdx.x
  int lo = 0, hi = a.n_utt - 1;
  const long long b = blockIdx.x;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (a.utts[mid].tile_begin <= b) lo = mid;
    else hi = mid - 1;
  }
  const ResampleUtt u = a.utts[lo];
  const In* in = static_cast<const In*>(a.in) + u.in_off;
  const long long n_out = (u.in_len * a.up + a.down - 1) / a.down;
  const long long m0 = (b - u.tile_begin) * 2 * a.H;
  const long long kb = (m0 * a.down + a.half) / a.up;          // the newest input of output m0
  const long long klo = kb - (a.K - 1);
  const long long qd = static_cast<long long>(a.q) * a.down;   // output m + H reads qd samples later
  // window: z[k] = (x[klo + k], x[klo + k + qd]), zero outside the utterance
  for (int k = tid; k < a.win; k += kResampleThreads) {
    const long long s0 = klo + k, s1 = s0 + qd;
    const float x0 = (s0 >= 0 && s0 < u.in_len) ? resample_load(in, s0) : 0.0f;
    const float x1 = (s1 >= 0 && s1 < u.in_len) ? resample_load(in, s1) : 0.0f;
    s_z[k] = make_float2(x0, x1);
  }
  for (int k = tid; k < a.up * a.Ks; k += kResampleThreads) s_taps[k] = a.taps[k];
  __syncthreads();
  for (int j = tid; j < a.H; j += kResampleThreads) {
    const long long t = (m0 + j) * a.down + a.half;
    const int p = static_cast<int>(t % a.up);
    const float2* z = s_z + static_cast<int>(t / a.up - klo);
    const float* hr = s_taps + p * a.Ks;
    float2 acc = make_float2(0.0f, 0.0f);
#pragma unroll 4
    for (int i = 0; i < a.K; ++i) {
      const float hv = hr[i];
      acc = __ffma2_rn(make_float2(hv, hv), z[-i], acc);
    }
    s_out[j] = static_cast<int16_t>(min(max(__float2int_rn(acc.x), -32768), 32767));
    s_out[j + a.H] = static_cast<int16_t>(min(max(__float2int_rn(acc.y), -32768), 32767));
  }
  __syncthreads();
  const long long cnt = min(static_cast<long long>(2 * a.H), n_out - m0);
  int16_t* out = a.out + u.out_off + m0;
  if (((u.out_off + m0) & 7) == 0) {   // 16-byte stores (d_out is 16-byte aligned)
    const int nv = static_cast<int>(cnt >> 3);
    for (int k = tid; k < nv; k += kResampleThreads)
      reinterpret_cast<int4*>(out)[k] = reinterpret_cast<const int4*>(s_out)[k];
    for (int k = nv * 8 + tid; k < cnt; k += kResampleThreads) out[k] = s_out[k];
  } else {
    for (int k = tid; k < cnt; k += kResampleThreads) out[k] = s_out[k];
  }
}

// ---- decode ----------------------------------------------------------------------------------------------------
template <int FMT>
__device__ __forceinline__ float pcm_value(const uint8_t* p, int be) {
  if constexpr (FMT == kPcmU8) {
    return static_cast<float>((static_cast<int>(p[0]) - 128) * 256);
  } else if constexpr (FMT == kPcmS16) {
    uint32_t v = *reinterpret_cast<const uint16_t*>(p);
    if (be) v = __byte_perm(v, 0, 0x3201);
    return static_cast<float>(static_cast<int16_t>(v));
  } else if constexpr (FMT == kPcmS24) {
    const uint32_t b0 = p[0], b1 = p[1], b2 = p[2];
    const uint32_t v = be ? (b0 << 24) | (b1 << 16) | (b2 << 8) : (b2 << 24) | (b1 << 16) | (b0 << 8);
    return static_cast<float>(static_cast<int32_t>(v) >> 8) * (1.0f / 256.0f);
  } else if constexpr (FMT == kPcmS32) {
    uint32_t v = *reinterpret_cast<const uint32_t*>(p);
    if (be) v = __byte_perm(v, 0, 0x0123);
    return static_cast<float>(static_cast<int32_t>(v)) * (1.0f / 65536.0f);
  } else if constexpr (FMT == kPcmF32) {
    uint32_t v = *reinterpret_cast<const uint32_t*>(p);
    if (be) v = __byte_perm(v, 0, 0x0123);
    const float x = __uint_as_float(v);
    return isfinite(x) ? x * 32768.0f : 0.0f;
  } else {
    unsigned long long v = *reinterpret_cast<const unsigned long long*>(p);
    if (be) {
      const uint32_t lo = static_cast<uint32_t>(v), hi = static_cast<uint32_t>(v >> 32);
      v = (static_cast<unsigned long long>(__byte_perm(lo, 0, 0x0123)) << 32) | __byte_perm(hi, 0, 0x0123);
    }
    const double x = __longlong_as_double(static_cast<long long>(v));
    return isfinite(x) ? static_cast<float>(x * 32768.0) : 0.0f;
  }
}

// Segment i turns frames src[i] .. src[i] + len[i] of the raw stream into dst[dst_off[i] ...]: the channels of a
// frame are summed in order in float32, then divided by C.
template <int FMT>
__global__ void __launch_bounds__(256) decode_pcm_kernel(const uint8_t* raw, int channels, int be, const long long* src,
                                                         const long long* dst_off, const long long* len, float* dst) {
  const int seg = blockIdx.y;
  const long long n = len[seg];
  const int fb = kPcmSize<FMT> * channels;
  const uint8_t* in = raw + src[seg] * fb;
  float* out = dst + dst_off[seg];
  const float fc = static_cast<float>(channels);
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long k = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; k < n; k += stride) {
    const uint8_t* f = in + k * fb;
    float s = pcm_value<FMT>(f, be);
    for (int c = 1; c < channels; ++c) s += pcm_value<FMT>(f + c * kPcmSize<FMT>, be);
    out[k] = channels == 1 ? s : s / fc;
  }
}
#endif  // VADB_RESAMPLE_KERNELS

}  // namespace vadb
