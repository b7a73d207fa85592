// vad_stream_resample.h -- index math of the resampling ragged bank (vadb200_stream_bank_create_ragged_rate): which
// 16 kHz samples a feed of source-rate samples makes ready, the tiles they are computed in, each tile's input window
// and where a source sample sits in the stream's history.  Plain C++ marked __host__ __device__:
// vad_stream_resample.cu's kernels use it, and tests/emul/emul_stream_resample.cpp drives the same functions on the
// host.
//
// The filter is vadb200_resample_packed's (vad_resample.cuh): output m reads the K source samples
// x[kb - K + 1 .. kb], kb = (m down + half) div up, against polyphase row (m down + half) mod up.  A stream that has
// taken N source samples since its last reset or end has produced the outputs whose newest input kb is below N:
// M(N) of them, the causal prefix of scipy.signal.resample_poly, which no later sample changes.  Output M(N) has
// kb >= N, so the outputs a feed of c samples adds, M(N) .. M(N + c) - 1, read nothing older than x[N - K + 1]: the
// stream keeps its last K - 1 source samples (zeros before its first) as history, slot k holding x[N - K + 1 + k].
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define VADB_SRS_HD __host__ __device__ __forceinline__
#else
#define VADB_SRS_HD inline
#endif

namespace vadb {

constexpr int kSrsTile = 256;   // 16 kHz outputs per tile (one per thread of stream_resample_kernel)

// M(N): outputs ready after n source samples.
VADB_SRS_HD long long srs_ready(long long n, int up, int down, int half) {
  const long long t = n * up - 1 - half;
  return t < 0 ? 0 : t / down + 1;
}
// kb: the newest source sample output m reads.
VADB_SRS_HD long long srs_newest(long long m, int up, int down, int half) {
  return (m * down + half) / up;
}
// cap16: the most outputs one feed of at most cap source samples adds (ceil(cap up / down); reached for some N).
VADB_SRS_HD int srs_cap16(int cap, int up, int down) {
  return static_cast<int>((static_cast<long long>(cap) * up + down - 1) / down);
}
// Tiles of a feed of c samples that adds `outs` outputs: ceil(outs / kSrsTile), and one for a packet that adds no
// output, since the last tile also writes the new history.  A stream with nothing new has none.
VADB_SRS_HD int srs_tiles(int c, int outs) {
  return c <= 0 ? 0 : outs > 0 ? (outs + kSrsTile - 1) / kSrsTile : 1;
}
// Source samples a tile stages: its outputs' inputs, and for the last tile everything up to the packet's end (the new
// history is the last K - 1 of them).  [lo, hi] in stream sample indices; ma < mb are the tile's outputs, and
// ma == mb for a packet that adds none.
struct SrsWindow {
  long long lo, hi;
};
VADB_SRS_HD SrsWindow srs_window(long long ma, long long mb, bool last, long long n_end, int up, int down, int half,
                                 int K) {
  SrsWindow w;
  w.lo = mb > ma ? srs_newest(ma, up, down, half) - (K - 1) : n_end - (K - 1);
  w.hi = last ? n_end - 1 : srs_newest(mb - 1, up, down, half);
  return w;
}
// The most entries a window holds: (kSrsTile - 1) outputs span (kSrsTile - 1) down / up + 1 samples, the last tile
// reaches at most ceil(down / up) - 1 samples past its last output's newest, plus the K - 1 older taps.
VADB_SRS_HD int srs_window_max(int up, int down, int K) {
  return static_cast<int>(static_cast<long long>(kSrsTile - 1) * down / up) + (down + up - 1) / up + K;
}
// History slot of source sample g >= n - K + 1 for a stream that had taken n samples (g < n).
VADB_SRS_HD int srs_hist_slot(long long g, long long n, int K) { return static_cast<int>(g - n + (K - 1)); }

}  // namespace vadb
