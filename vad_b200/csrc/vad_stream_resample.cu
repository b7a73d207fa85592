// vad_stream_resample.cu -- the resampling ragged bank's kernels (DESIGN.md section 5.9), in a translation unit of
// their own so that no pre-existing kernel's code moves.  A feed of source-rate packets is two kernels here, then the
// 16 kHz ragged bank's unchanged stream_ragged_kernel on the packed 16 kHz samples they leave:
//
// stream_resample_plan_kernel (one CTA): reads the n + 1 source offsets once, checks each length, advances each
//   stream's source count N and flips its history buffer, and scans the streams' 16 kHz counts M(N + c) - M(N) into
//   packed offsets (a bad stream gets cap16 + 1 samples, so the ragged kernel reports -1 and reads none) and their
//   tile counts into tile offsets.
// stream_resample_kernel: CTAs loop over the feed's tiles of kSrsTile outputs of one stream (a stream that takes a
//   second of audio spreads over many CTAs), stage the tile's source window from the old history and the packet, and
//   run one output per thread: vadb200_resample_packed's FMA chain on the same float32 taps, so the same bits.  A
//   stream's last tile also writes its new history into the other buffer.
// vadb200.cu validates every argument and counts the launches; these functions only enqueue.
#include "vad_resample.cuh"
#include "vad_stream_resample.h"

#include <algorithm>

namespace vadb {

constexpr int kSrsPlanThreads = 1024;
constexpr int kSrsEndThreads = 256;

__global__ void __launch_bounds__(kSrsPlanThreads) stream_resample_plan_kernel(const StreamResampleParams p) {
  __shared__ long long s_end[kSrsPlanThreads];   // offsets[i + 1] of the chunk's streams
  __shared__ long long s_w16[32];                // per warp: inclusive scan of the 16 kHz counts
  __shared__ int s_wt[32];                       //           and of the tile counts
  __shared__ long long s_base16, s_start;
  __shared__ int s_baset;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    s_base16 = 0;
    s_baset = 0;
    s_start = p.offsets[0];
  }
  for (int c0 = 0; c0 < p.n; c0 += kSrsPlanThreads) {
    const int i = c0 + tid;
    const int nloc = min(kSrsPlanThreads, p.n - c0);
    if (tid < nloc) s_end[tid] = p.offsets[i + 1];
    __syncthreads();
    long long len16 = 0;
    int tiles = 0;
    SrsFeed f{};
    if (tid < nloc) {
      const long long a = tid ? s_end[tid - 1] : s_start;
      const long long c = s_end[tid] - a;
      f.src = a;
      if (c < 0 || c > p.cap) {
        len16 = p.cap16 + 1;   // not advanced; stream_ragged_kernel reports -1
      } else {
        f.c = static_cast<int>(c);
        f.n0 = p.n_in[i];
        f.outs = static_cast<int>(srs_ready(f.n0 + c, p.up, p.down, p.half) - srs_ready(f.n0, p.up, p.down, p.half));
        f.rd = p.cur[i];
        len16 = f.outs;
        tiles = srs_tiles(f.c, f.outs);
        if (c > 0) {
          p.n_in[i] = f.n0 + c;
          p.cur[i] = f.rd ^ 1;
        }
      }
    }
    long long x = len16;
    int y = tiles;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long xv = __shfl_up_sync(0xffffffffu, x, o);
      const int yv = __shfl_up_sync(0xffffffffu, y, o);
      if (lane >= o) {
        x += xv;
        y += yv;
      }
    }
    if (lane == 31) {
      s_w16[warp] = x;
      s_wt[warp] = y;
    }
    __syncthreads();
    if (warp == 0) {
      long long a = s_w16[lane];
      int b = s_wt[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const long long av = __shfl_up_sync(0xffffffffu, a, o);
        const int bv = __shfl_up_sync(0xffffffffu, b, o);
        if (lane >= o) {
          a += av;
          b += bv;
        }
      }
      s_w16[lane] = a;
      s_wt[lane] = b;
    }
    __syncthreads();
    if (tid < nloc) {
      f.out = s_base16 + (warp ? s_w16[warp - 1] : 0) + x - len16;
      p.off16[i] = f.out;
      p.tile_off[i] = s_baset + (warp ? s_wt[warp - 1] : 0) + y - tiles;
      p.feed[i] = f;
    }
    __syncthreads();
    if (tid == 0) {
      s_base16 += s_w16[31];
      s_baset += s_wt[31];
      s_start = s_end[nloc - 1];
    }
    __syncthreads();
  }
  if (tid == 0) {
    p.off16[p.n] = s_base16;
    p.tile_off[p.n] = s_baset;
  }
}

__global__ void __launch_bounds__(kSrsTile) stream_resample_kernel(const StreamResampleParams p) {
  extern __shared__ float s_x[];   // the tile's source window, x[w.lo + k]
  const int tid = threadIdx.x;
  const int total = p.tile_off[p.n];
  for (int t = blockIdx.x; t < total; t += gridDim.x) {
    // stream of this tile: the last one whose first tile is <= t (it has tiles, so it is the only such one with any)
    int lo = 0, hi = p.n - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (p.tile_off[mid] <= t) lo = mid;
      else hi = mid - 1;
    }
    const SrsFeed f = p.feed[lo];
    const bool last = t == p.tile_off[lo + 1] - 1;
    const long long m0 = srs_ready(f.n0, p.up, p.down, p.half);
    const long long ma = m0 + static_cast<long long>(t - p.tile_off[lo]) * kSrsTile;
    const long long mb = min(ma + kSrsTile, m0 + f.outs);
    const long long n_end = f.n0 + f.c;
    const SrsWindow w = srs_window(ma, mb, last, n_end, p.up, p.down, p.half, p.K);
    const int nw = static_cast<int>(w.hi - w.lo + 1);
    const int16_t* old = p.hist + (static_cast<long long>(f.rd) * p.n + lo) * p.hs;
    for (int k = tid; k < nw; k += kSrsTile) {
      const long long g = w.lo + k;
      const int v = g < f.n0 ? old[srs_hist_slot(g, f.n0, p.K)] : p.samples[f.src + (g - f.n0)];
      s_x[k] = static_cast<float>(v);
    }
    __syncthreads();
    const long long m = ma + tid;
    if (m < mb) {
      const long long tt = m * p.down + p.half;
      const float* hr = p.taps + static_cast<int>(tt % p.up) * p.Ks;
      const float* z = s_x + static_cast<int>(tt / p.up - w.lo);
      float acc = 0.0f;
#pragma unroll 4
      for (int i = 0; i < p.K; ++i) acc = __fmaf_rn(__ldg(hr + i), z[-i], acc);
      p.pcm16[f.out + (m - m0)] = static_cast<int16_t>(min(max(__float2int_rn(acc), -32768), 32767));
    }
    if (last) {   // the new history: x[n_end - K + 1 .. n_end - 1], zeros before the stream's first sample
      int16_t* nh = p.hist + (static_cast<long long>(f.rd ^ 1) * p.n + lo) * p.hs;
      const int k0 = static_cast<int>(n_end - (p.K - 1) - w.lo);
      for (int k = tid; k < p.hs; k += kSrsTile) nh[k] = static_cast<int16_t>(static_cast<int>(s_x[k0 + k]));
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kSrsEndThreads) stream_resample_end_kernel(const StreamResampleParams p,
                                                                           const uint8_t* end) {
  const long long per = 2LL * p.hs + 1;
  const long long q = static_cast<long long>(blockIdx.x) * kSrsEndThreads + threadIdx.x;
  const long long i = q / per;
  if (i >= p.n || !end[i]) return;
  const int r = static_cast<int>(q - i * per);
  if (r == 2 * p.hs) {
    p.n_in[i] = 0;
  } else {
    const int b = r / p.hs, k = r - b * p.hs;
    p.hist[(b * static_cast<long long>(p.n) + i) * p.hs + k] = 0;
  }
}

void enqueue_stream_resample(const StreamResampleParams& p, int grid, cudaStream_t st) {
  stream_resample_plan_kernel<<<1, kSrsPlanThreads, 0, st>>>(p);
  const size_t smem = static_cast<size_t>(srs_window_max(p.up, p.down, p.K)) * sizeof(float);
  stream_resample_kernel<<<grid, kSrsTile, smem, st>>>(p);
}

void enqueue_stream_resample_end(const StreamResampleParams& p, const uint8_t* end, cudaStream_t st) {
  const long long work = static_cast<long long>(p.n) * (2LL * p.hs + 1);
  stream_resample_end_kernel<<<static_cast<unsigned>((work + kSrsEndThreads - 1) / kSrsEndThreads), kSrsEndThreads,
                               0, st>>>(p, end);
}

}  // namespace vadb
