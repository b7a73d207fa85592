// vad_segments.cuh -- frame decisions -> smoothed labels -> speech segments -> speech-only PCM (sm_100a).
//
// Semantics (this project's own definition; oracle/ref_segments.py restates it sequentially over runs).  Per
// utterance, over its R = T - 5 label rows (nonzero = speech), in this order:
//   1. gap filling:   a maximal non-speech run with speech on both sides, shorter than G = min_silence_rows,
//                     becomes speech (runs touching an utterance edge are never filled);
//   2. short runs:    a maximal speech run shorter than S = min_speech_rows becomes non-speech;
//   3. padding:       a row becomes speech when a speech row lies within P = pad_rows of it.
// G <= 1, S <= 1 and P == 0 switch their step off.  A segment is a maximal smoothed speech run [r0, r1) and maps
// to the samples [160 r0 + 440, 160 r1 + 440) of its utterance: row r classifies frame r + 2 and owns that frame's
// centre hop.
//
// Bounded window.  Each row's result depends only on rows within H = (G - 1) + (S - 1) + P of it, so the
// smoothing kernel works on tiles of at most kSpeechTile rows of one utterance, loaded with a halo of H rows (one
// more on the left, for the row before the tile) and clipped to the utterance.  A window edge that is not an
// utterance edge can only lose a gap fill at distance >= G - 1 or shorten a run whose stretch inside the window
// is already >= S long, so every row the tile writes is exact.  Within a window each thread owns one contiguous
// chunk; the three steps need, per row, the nearest marked row on each side (speech for steps 1 and 3,
// non-speech for step 2), which is a serial pass over the chunk seeded by one block-wide max / min scan of the
// chunks' edge positions.  All cross-chunk information travels through those scans.
//
// The per-thread functions are plain C++ marked __host__ __device__: the kernels inline them and
// tests/emul/emul_segments.cpp drives them on the host through the same tile, halo and chunk index math.
#pragma once

#include <cstdint>

#include "vad_ragged.h"

#if defined(__CUDACC__)
#define VADB_SEG_HD __host__ __device__ __forceinline__
#else
#define VADB_SEG_HD inline
#endif

namespace vadb {

constexpr int kSpeechTile = 2048;          // rows of one utterance per smoothing / segment CTA
constexpr int kSpeechThreads = 256;        // threads of the smoothing, segment and gather kernels
constexpr int kSpeechMaxParam = 1000;      // rows (10 s) per parameter
constexpr int kSpeechHopSamples = 160;     // one row's hop
constexpr int kSpeechFirstSample = 440;    // row 0 owns samples [440, 600): centre hop of frame 2
constexpr int kSpeechScanThreads = 1024;   // single-CTA scan over the tile counts
constexpr int kSpeechScanPer = 8;          // tile counts per scan thread and pass

// One smoothing tile: rows [r0, r0 + n) of utterance u (global row indices).
struct SpeechTile {
  long long r0;
  int n;
  int u;
};

// The step parameters as they reach the kernels: each step's halo contribution is 0 when the step is off.
struct SmoothParams {
  int G, S, P;  // min_silence_rows, min_speech_rows, pad_rows
  int H;        // (G > 1 ? G - 1 : 0) + (S > 1 ? S - 1 : 0) + P
};

VADB_SEG_HD SmoothParams smooth_params(int min_speech_rows, int min_silence_rows, int pad_rows) {
  SmoothParams sp;
  sp.G = min_silence_rows;
  sp.S = min_speech_rows;
  sp.P = pad_rows;
  sp.H = (sp.G > 1 ? sp.G - 1 : 0) + (sp.S > 1 ? sp.S - 1 : 0) + sp.P;
  return sp;
}

// Window of one tile: global rows [w0, w0 + n); the tile's rows are window rows [t0, o1); o0 = t0 - 1 when the
// tile does not start its utterance (the row before it decides whether the tile's first row starts a segment).
struct SmoothWindow {
  long long w0;
  int n, o0, t0, o1;
};

VADB_SEG_HD SmoothWindow smooth_window(const SpeechTile& t, long long ubeg, long long uend, int H) {
  SmoothWindow w;
  const long long lo = t.r0 - H - 1, hi = t.r0 + t.n + H;
  w.w0 = lo > ubeg ? lo : ubeg;
  const long long w1 = hi < uend ? hi : uend;
  w.n = static_cast<int>(w1 - w.w0);
  w.t0 = static_cast<int>(t.r0 - w.w0);
  w.o0 = t.r0 > ubeg ? w.t0 - 1 : w.t0;
  w.o1 = w.t0 + t.n;
  return w;
}

// Largest window a launch can see; the smoothing kernel's shared memory is 4 bytes per window row.
VADB_SEG_HD int smooth_window_cap(int H) { return kSpeechTile + 2 * H + 1; }
VADB_SEG_HD int smooth_smem_bytes(int H) { return 4 * ((smooth_window_cap(H) + 15) & ~15); }

// Thread `tid`'s chunk of a window of n rows: [c0, c1).
VADB_SEG_HD void smooth_chunk(int n, int tid, int& c0, int& c1) {
  const int c = (n + kSpeechThreads - 1) / kSpeechThreads;
  c0 = tid * c;
  c1 = c0 + c < n ? c0 + c : n;
  if (c0 > n) c0 = n;
}

// Load the window's labels as 0/1 into a[] and return the chunk's outermost speech rows (last / first; -1 / n
// when the chunk has none).
VADB_SEG_HD void smooth_load(const uint8_t* labels, long long w0, int n, int c0, int c1, uint8_t* a, int& last,
                             int& first) {
  last = -1;
  first = n;
  for (int i = c0; i < c1; ++i) {
    const uint8_t v = labels[w0 + i] != 0;
    a[i] = v;
    if (v) {
      last = i;
      if (first == n) first = i;
    }
  }
}

// Outermost rows of the chunk whose value equals `want`.
VADB_SEG_HD void smooth_edges(const uint8_t* x, int n, int c0, int c1, uint8_t want, int& last, int& first) {
  last = -1;
  first = n;
  for (int i = c0; i < c1; ++i)
    if (x[i] == want) {
      last = i;
      if (first == n) first = i;
    }
}

// Step 1.  lin = last speech row before the chunk (-1: none in the window), rin = first after it (n: none).
// b[i] = a[i], or 1 when row i lies in a non-speech run bounded by speech on both sides and shorter than G.
VADB_SEG_HD void smooth_fill(const uint8_t* a, uint8_t* b, int16_t* prv, int n, int c0, int c1, int lin, int rin,
                             int G) {
  int p = lin;
  for (int i = c0; i < c1; ++i) {
    if (a[i]) p = i;
    prv[i] = static_cast<int16_t>(p);
  }
  int q = rin;
  for (int i = c1 - 1; i >= c0; --i) {
    if (a[i]) {
      q = i;
      b[i] = 1;
    } else {
      const int pi = prv[i];
      b[i] = (G > 1 && pi >= 0 && q < n && q - pi - 1 < G) ? 1 : 0;
    }
  }
}

// Step 2.  lin / rin: last / first NON-speech row of b outside the chunk (-1 / n: the window edge bounds the run).
// a[i] = b[i] unless row i's speech run is shorter than S.
VADB_SEG_HD void smooth_runs(const uint8_t* b, uint8_t* a, int16_t* prv, int c0, int c1, int lin, int rin, int S) {
  int p = lin;
  for (int i = c0; i < c1; ++i) {
    if (!b[i]) p = i;
    prv[i] = static_cast<int16_t>(p);
  }
  int q = rin;
  for (int i = c1 - 1; i >= c0; --i) {
    if (!b[i]) {
      q = i;
      a[i] = 0;
    } else {
      a[i] = (S <= 1 || q - prv[i] - 1 >= S) ? 1 : 0;
    }
  }
}

// Step 3 over the output rows [o0, o1) of the chunk: b[i] = 1 when a speech row of a lies within P of row i.
// lin / rin: last / first speech row of a outside the chunk.
VADB_SEG_HD void smooth_pad(const uint8_t* a, uint8_t* b, int16_t* prv, int n, int c0, int c1, int lin, int rin,
                            int P, int o0, int o1) {
  int p = lin;
  for (int i = c0; i < c1; ++i) {
    if (a[i]) p = i;
    prv[i] = static_cast<int16_t>(p);
  }
  int q = rin;
  for (int i = c1 - 1; i >= c0; --i) {
    if (a[i]) q = i;
    if (i >= o0 && i < o1) {
      const int pi = prv[i];
      b[i] = ((pi >= 0 && i - pi <= P) || (q < n && q - i <= P)) ? 1 : 0;
    }
  }
}

// Row i of the tile (window row, t0 <= i < o1) starts a segment; s[] holds the smoothed rows [o0, o1).
VADB_SEG_HD bool seg_starts(const uint8_t* s, int o0, int i) { return s[i] && (i == o0 || !s[i - 1]); }

// Samples of a segment [r0, r1) within its utterance.
VADB_SEG_HD long long seg_sample(long long r) { return kSpeechHopSamples * r + kSpeechFirstSample; }

// ---- online smoothing for the stream bank -------------------------------------------------------------------
// The same three steps as a causal cascade, one row in per tick.  Step 1 (gap fill) holds its last d1 = G - 1 rows
// (G > 1, else it passes rows through) in a bit ring, the length of the trailing non-speech run and whether speech
// was seen; when speech ends a non-speech run shorter than G that has speech before it, it sets the run's bits.
// Step 2 (short runs) holds d2 = S - 1 rows and the trailing speech run; when a run shorter than S ends it clears
// the run's bits.  Step 3 (pad) needs no ring: its row q is speech iff its last speech input lies at or after q - P.
// Each step emits its oldest row once its ring is full, so after the first H = d1 + d2 + P rows the cascade emits
// exactly one row per row fed: row r is final when row r + H arrives.  At the end of a stream the steps drain in
// order with the offline edge rules: a trailing silence is never filled, a trailing speech run is judged with the
// length it has, and the pad is clipped.
//
// State, struct-of-arrays over streams (word k of stream s at [k * n + s]): ring1 [W1][n], ring2 [W2][n] with
// W = ceil(d / 32), meta [n] and last [n]; all zero is a fresh stream.  A ring slot of input row t is t mod d.
constexpr uint32_t kSegRunMask = 0x7ffu;  // run lengths are clamped to <= 1000 < 2^11
constexpr int kSegSeenBit = 11;           // step 1 has seen speech
constexpr int kSegRun2Shift = 12;         // step 2's trailing speech run
constexpr int kSegOutBit = 23;            // the last emitted row (a segment is open)
constexpr int kSegEndThreads = 128;       // streams per CTA of stream_end_kernel

struct StreamSeg {
  uint32_t* ring1;
  uint32_t* ring2;
  uint32_t* meta;  // step 1's trailing non-speech run | seen | step 2's trailing speech run | last emitted row
  int* last;       // step 3's last speech input + 1 (0: none)
  long long n;     // streams (the SoA stride)
  int G, S, P, d1, d2, H;
  uint8_t* rows;    // [n] finalised row per feed, nullable
  int64_t* bounds;  // [n] its segment bound, nullable
};

VADB_SEG_HD int seg_ring_words(int d) { return (d + 31) >> 5; }

VADB_SEG_HD int ring_get(const uint32_t* ring, long long stride, int slot) {
  return static_cast<int>((ring[(slot >> 5) * stride] >> (slot & 31)) & 1u);
}

// Set (v = 1) or clear slots [a, b) of a ring, 0 <= a < b <= 32 W.
VADB_SEG_HD void ring_span(uint32_t* ring, long long stride, int a, int b, int v) {
  for (int w = a >> 5; w <= (b - 1) >> 5; ++w) {
    const int lo = (a > 32 * w ? a : 32 * w) - 32 * w, hi = (b < 32 * w + 32 ? b : 32 * w + 32) - 32 * w;
    const uint32_t m = (hi - lo == 32 ? 0xffffffffu : ((1u << (hi - lo)) - 1u)) << lo;
    uint32_t& x = ring[w * stride];
    x = v ? (x | m) : (x & ~m);
  }
}

// Set or clear the `len` rows just before the row whose slot is `end` (0 < len <= d): one or two spans.
VADB_SEG_HD void ring_run(uint32_t* ring, long long stride, int d, int end, int len, int v) {
  const int a = end >= len ? end - len : end - len + d;
  if (a + len <= d) {
    ring_span(ring, stride, a, a + len, v);
  } else {
    ring_span(ring, stride, a, d, v);
    ring_span(ring, stride, 0, a + len - d, v);
  }
}

// Push row t (value v) into a ring of d > 0 rows; returns its oldest row t - d, or -1 while t < d.
VADB_SEG_HD int ring_push(uint32_t* ring, long long stride, int d, int t, int v) {
  const int slot = t % d;
  const int out = t >= d ? ring_get(ring, stride, slot) : -1;
  uint32_t& x = ring[(slot >> 5) * stride];
  x = (x & ~(1u << (slot & 31))) | (static_cast<uint32_t>(v) << (slot & 31));
  return out;
}

// Step 1, input row t of a stream: returns step 1's output row t - d1 (-1: none yet).
VADB_SEG_HD int seg_fill_push(const StreamSeg& g, uint32_t* ring, long long stride, int t, int v, uint32_t& meta) {
  if (g.d1 == 0) return v;
  uint32_t z = meta & kSegRunMask;
  if (v) {
    if (z > 0 && ((meta >> kSegSeenBit) & 1u) && z < static_cast<uint32_t>(g.G))
      ring_run(ring, stride, g.d1, t % g.d1, static_cast<int>(z), 1);
    z = 0;
    meta |= 1u << kSegSeenBit;
  } else if (z < static_cast<uint32_t>(g.G)) {
    ++z;
  }
  meta = (meta & ~kSegRunMask) | z;
  return ring_push(ring, stride, g.d1, t, v);
}

// Step 2, input row t: returns its output row t - d2 (-1: none yet).  A short run ends on a non-speech row.
VADB_SEG_HD int seg_runs_push(const StreamSeg& g, uint32_t* ring, long long stride, int t, int v, uint32_t& meta) {
  if (g.d2 == 0) return v;
  uint32_t run = (meta >> kSegRun2Shift) & kSegRunMask;
  if (v) {
    if (run < static_cast<uint32_t>(g.S)) ++run;
  } else {
    if (run > 0 && run < static_cast<uint32_t>(g.S)) ring_run(ring, stride, g.d2, t % g.d2, static_cast<int>(run), 0);
    run = 0;
  }
  meta = (meta & ~(kSegRunMask << kSegRun2Shift)) | (run << kSegRun2Shift);
  return ring_push(ring, stride, g.d2, t, v);
}

// Step 3's row q: speech iff its last speech input (last - 1) lies at or after q - P.
VADB_SEG_HD int seg_pad_row(int q, int P, int last) { return last > 0 && last - 1 >= q - P ? 1 : 0; }

// Emitted row q with value y: its bound (160 q + 440 when it opens or closes a segment, else -1).
VADB_SEG_HD long long seg_emit(int q, int y, uint32_t& meta) {
  const int prev = static_cast<int>((meta >> kSegOutBit) & 1u);
  meta = (meta & ~(1u << kSegOutBit)) | (static_cast<uint32_t>(y) << kSegOutBit);
  return y != prev ? seg_sample(q) : -1;
}

// One row r (value v != 0: speech) of stream s.  Returns the row it finalises, r - H (-1: none), with its value
// and bound.
VADB_SEG_HD int seg_step(const StreamSeg& g, long long s, int r, int v, uint8_t& row, long long& bound) {
  uint32_t meta = g.meta[s];
  int q = -1;
  row = 255;
  bound = -1;
  int x = seg_fill_push(g, g.ring1 + s, g.n, r, v, meta);
  if (x >= 0) x = seg_runs_push(g, g.ring2 + s, g.n, r - g.d1, x, meta);
  if (x >= 0) {
    const int t3 = r - g.d1 - g.d2;
    int last = g.last[s];
    if (x) g.last[s] = last = t3 + 1;
    if (t3 >= g.P) {
      q = t3 - g.P;
      const int y = seg_pad_row(q, g.P, last);
      row = static_cast<uint8_t>(y);
      bound = seg_emit(q, y, meta);
    }
  }
  g.meta[s] = meta;
  return q;
}

// End of a stream that took R rows: emit(q, value, bound) for its min(R, H) pending rows in order; returns the
// close of a segment still open (160 R + 440) or -1.  Rings are read and written through (ring1, ring2, stride),
// which may be a copy of the stream's state; meta and last are the stream's values, updated in place.
template <class Emit>
VADB_SEG_HD long long seg_drain(const StreamSeg& g, uint32_t* ring1, uint32_t* ring2, long long stride, int R,
                                uint32_t& meta, int& last, Emit emit) {
  int t2 = R - g.d1 > 0 ? R - g.d1 : 0;
  int t3 = t2 - g.d2 > 0 ? t2 - g.d2 : 0;
  auto pad_in = [&](int x) {
    if (x) last = t3 + 1;
    if (t3 >= g.P) {
      const int q = t3 - g.P, y = seg_pad_row(q, g.P, last);
      emit(q, y, seg_emit(q, y, meta));
    }
    ++t3;
  };
  auto runs_in = [&](int x) {
    const int y = seg_runs_push(g, ring2, stride, t2++, x, meta);
    if (y >= 0) pad_in(y);
  };
  if (g.d1 > 0)  // step 1: the rows still held, unfilled
    for (int p = R - g.d1 > 0 ? R - g.d1 : 0; p < R; ++p) runs_in(ring_get(ring1, stride, p % g.d1));
  if (g.d2 > 0) {  // step 2: the trailing run counts with the length it has
    const uint32_t run = (meta >> kSegRun2Shift) & kSegRunMask;
    if (run > 0 && run < static_cast<uint32_t>(g.S)) ring_run(ring2, stride, g.d2, t2 % g.d2, static_cast<int>(run), 0);
    for (int p = t2 - g.d2 > 0 ? t2 - g.d2 : 0; p < t2; ++p) pad_in(ring_get(ring2, stride, p % g.d2));
  }
  for (int q = t3 - g.P > 0 ? t3 - g.P : 0; q < t3; ++q) {  // step 3: the pad clipped at row R
    const int y = seg_pad_row(q, g.P, last);
    emit(q, y, seg_emit(q, y, meta));
  }
  return (meta >> kSegOutBit) & 1u ? seg_sample(R) : -1;
}

// End stream s after R rows: its rings move to scratch (word k at scratch[k * sstride]) and the drain runs there;
// tail_rows [n][H] gets the pending rows then 255, tail_bounds [n][H + 1] their bounds, the close, then -1 (both
// nullable).  The stream's segment state is zero afterwards.
VADB_SEG_HD void seg_end(const StreamSeg& g, long long s, int R, uint32_t* scratch, long long sstride,
                         uint8_t* tail_rows, int64_t* tail_bounds) {
  const int w1 = g.d1 > 0 ? seg_ring_words(g.d1) : 0, w2 = g.d2 > 0 ? seg_ring_words(g.d2) : 0;
  for (int k = 0; k < w1; ++k) {
    scratch[k * sstride] = g.ring1[k * g.n + s];
    g.ring1[k * g.n + s] = 0;
  }
  for (int k = 0; k < w2; ++k) {
    scratch[(w1 + k) * sstride] = g.ring2[k * g.n + s];
    g.ring2[k * g.n + s] = 0;
  }
  uint32_t meta = g.meta[s];
  int last = g.last[s];
  uint8_t* rows = tail_rows ? tail_rows + s * g.H : nullptr;
  int64_t* bounds = tail_bounds ? tail_bounds + s * (g.H + 1) : nullptr;
  int j = 0;
  const long long close = seg_drain(g, scratch, scratch + w1 * sstride, sstride, R, meta, last,
                                    [&](int, int y, long long b) {
                                      if (rows) rows[j] = static_cast<uint8_t>(y);
                                      if (bounds) bounds[j] = b;
                                      ++j;
                                    });
  if (rows)
    for (int k = j; k < g.H; ++k) rows[k] = 255;
  if (bounds)
    for (int k = j; k <= g.H; ++k) bounds[k] = k == j ? close : -1;
  g.meta[s] = 0;
  g.last[s] = 0;
}

#if defined(__CUDACC__)

// Exclusive max of `last` over lower threads (-1 for thread 0) and exclusive min of `first` over higher threads
// (n for the last thread).  sh: 2 * (kSpeechThreads / 32) ints.
__device__ __forceinline__ void speech_block_edges(int last, int first, int n, int* sh, int& lin, int& rin) {
  constexpr int kWarps = kSpeechThreads / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int il = last, ir = first;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int vl = __shfl_up_sync(0xffffffffu, il, d);
    const int vr = __shfl_down_sync(0xffffffffu, ir, d);
    if (lane >= d) il = il > vl ? il : vl;
    if (lane + d < 32) ir = ir < vr ? ir : vr;
  }
  if (lane == 31) sh[warp] = il;
  if (lane == 0) sh[kWarps + warp] = ir;
  __syncthreads();
  int el = __shfl_up_sync(0xffffffffu, il, 1);
  int er = __shfl_down_sync(0xffffffffu, ir, 1);
  if (lane == 0) el = -1;
  if (lane == 31) er = n;
  for (int w = 0; w < warp; ++w) el = el > sh[w] ? el : sh[w];
  for (int w = warp + 1; w < kWarps; ++w) er = er < sh[kWarps + w] ? er : sh[kWarps + w];
  __syncthreads();
  lin = el;
  rin = er;
}

// Exclusive block scan of two int64 sums; returns the block totals through tot0 / tot1.  sh: 2 * warps.
template <int kT>
__device__ __forceinline__ void speech_block_scan2(long long& x0, long long& x1, long long* sh, long long& tot0,
                                                   long long& tot1) {
  constexpr int kWarps = kT / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long i0 = x0, i1 = x1;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const long long v0 = __shfl_up_sync(0xffffffffu, i0, d);
    const long long v1 = __shfl_up_sync(0xffffffffu, i1, d);
    if (lane >= d) {
      i0 += v0;
      i1 += v1;
    }
  }
  if (lane == 31) {
    sh[warp] = i0;
    sh[kWarps + warp] = i1;
  }
  __syncthreads();
  long long b0 = 0, b1 = 0;
  tot0 = 0;
  tot1 = 0;
  for (int w = 0; w < kWarps; ++w) {
    if (w < warp) {
      b0 += sh[w];
      b1 += sh[kWarps + w];
    }
    tot0 += sh[w];
    tot1 += sh[kWarps + w];
  }
  __syncthreads();
  x0 = b0 + i0 - x0;
  x1 = b1 + i1 - x1;
}

// Kernel 1: one CTA per tile.  Writes the tile's smoothed rows and its (segment starts, speech rows).
__global__ void __launch_bounds__(kSpeechThreads) speech_smooth_kernel(
    const uint8_t* __restrict__ labels, const SpeechTile* __restrict__ tiles, const long long* __restrict__ row_off,
    SmoothParams sp, uint8_t* __restrict__ smoothed, int2* __restrict__ tile_counts) {
  extern __shared__ __align__(16) unsigned char seg_smem[];
  __shared__ int sh_edges[2 * (kSpeechThreads / 32)];
  __shared__ long long sh_sum[2 * (kSpeechThreads / 32)];
  const SpeechTile t = tiles[blockIdx.x];
  const long long ubeg = row_off[t.u], uend = row_off[t.u + 1];
  const SmoothWindow w = smooth_window(t, ubeg, uend, sp.H);
  const int cap = (smooth_window_cap(sp.H) + 15) & ~15;
  uint8_t* a = seg_smem;
  uint8_t* b = seg_smem + cap;
  int16_t* prv = reinterpret_cast<int16_t*>(seg_smem + 2 * cap);
  int c0, c1, last, first, lin, rin;
  smooth_chunk(w.n, threadIdx.x, c0, c1);
  smooth_load(labels, w.w0, w.n, c0, c1, a, last, first);
  speech_block_edges(last, first, w.n, sh_edges, lin, rin);
  smooth_fill(a, b, prv, w.n, c0, c1, lin, rin, sp.G);
  smooth_edges(b, w.n, c0, c1, 0, last, first);
  speech_block_edges(last, first, w.n, sh_edges, lin, rin);
  smooth_runs(b, a, prv, c0, c1, lin, rin, sp.S);
  smooth_edges(a, w.n, c0, c1, 1, last, first);
  speech_block_edges(last, first, w.n, sh_edges, lin, rin);
  smooth_pad(a, b, prv, w.n, c0, c1, lin, rin, sp.P, w.o0, w.o1);
  __syncthreads();
  long long starts = 0, speech = 0;
  for (int i = w.t0 + static_cast<int>(threadIdx.x); i < w.o1; i += kSpeechThreads) {
    const uint8_t v = b[i];
    smoothed[w.w0 + i] = v;
    speech += v;
    starts += seg_starts(b, w.o0, i);
  }
  long long tot0, tot1;
  speech_block_scan2<kSpeechThreads>(starts, speech, sh_sum, tot0, tot1);
  if (threadIdx.x == 0) tile_counts[blockIdx.x] = make_int2(static_cast<int>(tot0), static_cast<int>(tot1));
}

// Kernel 2: one CTA.  prefix[t] = (segments, speech rows) of the tiles before t, t = 0 .. n_tiles.
__global__ void __launch_bounds__(kSpeechScanThreads) speech_scan_kernel(const int2* __restrict__ tile_counts,
                                                                         int n_tiles, longlong2* __restrict__ prefix) {
  __shared__ long long sh[2 * (kSpeechScanThreads / 32)];
  long long c0 = 0, c1 = 0;
  constexpr int kPass = kSpeechScanThreads * kSpeechScanPer;
  for (int base = 0; base < n_tiles; base += kPass) {
    const int i0 = base + threadIdx.x * kSpeechScanPer;
    int2 v[kSpeechScanPer];
    long long s0 = 0, s1 = 0;
#pragma unroll
    for (int k = 0; k < kSpeechScanPer; ++k) {
      v[k] = i0 + k < n_tiles ? tile_counts[i0 + k] : make_int2(0, 0);
      s0 += v[k].x;
      s1 += v[k].y;
    }
    long long tot0, tot1;
    speech_block_scan2<kSpeechScanThreads>(s0, s1, sh, tot0, tot1);
    s0 += c0;
    s1 += c1;
#pragma unroll
    for (int k = 0; k < kSpeechScanPer; ++k) {
      if (i0 + k < n_tiles) prefix[i0 + k] = make_longlong2(s0, s1);
      s0 += v[k].x;
      s1 += v[k].y;
    }
    c0 += tot0;
    c1 += tot1;
  }
  if (threadIdx.x == 0) prefix[n_tiles] = make_longlong2(c0, c1);
}

// Kernel 3: CTAs below n_tiles write their tile's segments; every CTA writes the per-utterance offsets of
// utterances [blockIdx.x * kSpeechThreads, +kSpeechThreads) ∩ [0, n_utt].
__global__ void __launch_bounds__(kSpeechThreads) speech_segments_kernel(
    const uint8_t* __restrict__ smoothed, const SpeechTile* __restrict__ tiles, const long long* __restrict__ row_off,
    const longlong2* __restrict__ prefix, int n_tiles, const int* __restrict__ utt_tile, long long n_utt,
    long long* __restrict__ segments, long long* __restrict__ seg_off, long long* __restrict__ speech_off) {
  __shared__ uint8_t s[kSpeechTile + 2];
  __shared__ long long sh_sum[2 * (kSpeechThreads / 32)];
  const long long u = static_cast<long long>(blockIdx.x) * kSpeechThreads + threadIdx.x;
  if (u <= n_utt) {
    const longlong2 pf = prefix[utt_tile[u]];
    seg_off[u] = pf.x;
    if (speech_off) speech_off[u] = kSpeechHopSamples * pf.y;
  }
  if (static_cast<int>(blockIdx.x) >= n_tiles) return;
  const SpeechTile t = tiles[blockIdx.x];
  const long long ubeg = row_off[t.u], uend = row_off[t.u + 1];
  // s[j] = smoothed row t.r0 - 1 + j, j in [o0, n2): the row before the tile and the row after it when they exist
  const int o0 = t.r0 > ubeg ? 0 : 1;
  const int n2 = t.n + 1 + (t.r0 + t.n < uend ? 1 : 0);
  for (int j = o0 + threadIdx.x; j < n2; j += kSpeechThreads) s[j] = smoothed[t.r0 - 1 + j];
  __syncthreads();
  constexpr int kPer = kSpeechTile / kSpeechThreads;
  const int j0 = 1 + threadIdx.x * kPer, j1 = j0 + kPer < t.n + 1 ? j0 + kPer : t.n + 1;
  long long cnt = 0, dummy = 0;
  for (int j = j0; j < j1; ++j) cnt += seg_starts(s, o0, j);
  long long tot0, tot1;
  speech_block_scan2<kSpeechThreads>(cnt, dummy, sh_sum, tot0, tot1);
  long long k = prefix[blockIdx.x].x + cnt;  // segments started before row j (global index of the next one)
  for (int j = j0; j < j1; ++j) {
    if (!s[j]) continue;
    const long long r = t.r0 - 1 + j - ubeg;  // row within the utterance
    if (seg_starts(s, o0, j)) segments[2 * k++] = seg_sample(r);
    if (j + 1 == n2 || !s[j + 1]) segments[2 * (k - 1) + 1] = seg_sample(r + 1);
  }
}

// Kernel 4: speech PCM.  Output hops are split evenly over the grid; each CTA walks the segments of the
// utterance that holds its first output hop in batches of kSpeechThreads (one segment per thread, an exclusive
// scan of their lengths gives their output positions) and copies the part of each batch that falls in its hop
// range with 16-byte loads and stores.  Segment starts, utterance offsets and output positions are multiples of
// 8 samples, so every 8-sample vector lies in one hop of one segment.
constexpr int kGatherUnroll = 4;

__global__ void __launch_bounds__(kSpeechThreads) speech_gather_kernel(
    const int16_t* __restrict__ pcm, const long long* __restrict__ utt_off, long long n_utt,
    const long long* __restrict__ segments, const long long* __restrict__ seg_off,
    const long long* __restrict__ speech_off, int16_t* __restrict__ out, long long out_capacity) {
  __shared__ long long s_dst[kSpeechThreads + 1];  // output sample of each batch segment, then the batch end
  __shared__ long long s_src[kSpeechThreads];      // pcm index minus output index for each batch segment
  __shared__ long long sh_sum[2 * (kSpeechThreads / 32)];
  __shared__ long long s_u;
  const long long total = speech_off[n_utt];
  const long long hops = total / kSpeechHopSamples;
  const long long h0 = hops * blockIdx.x / gridDim.x, h1 = hops * (blockIdx.x + 1) / gridDim.x;
  if (h0 >= h1) return;
  const long long lo = kSpeechHopSamples * h0;
  const long long hi_s = kSpeechHopSamples * h1 < out_capacity ? kSpeechHopSamples * h1 : out_capacity;
  if (lo >= hi_s) return;
  if (threadIdx.x == 0) {  // utterance holding output sample lo: last u with speech_off[u] <= lo
    long long a = 0, b = n_utt;  // speech_off[a] <= lo < speech_off[b]
    while (b - a > 1) {
      const long long m = (a + b) >> 1;
      if (speech_off[m] <= lo) a = m; else b = m;
    }
    s_u = a;
  }
  __syncthreads();
  const long long u0 = s_u;
  const long long n_seg = seg_off[n_utt];
  long long j = seg_off[u0], dst = speech_off[u0];
  while (dst < hi_s && j < n_seg) {
    const long long jj = j + threadIdx.x;
    long long len = 0, zero = 0, src = 0;
    if (jj < n_seg) {
      const long long sb = segments[2 * jj], se = segments[2 * jj + 1];
      len = se - sb;
      long long a = u0, b = n_utt;  // utterance of segment jj: last u with seg_off[u] <= jj
      while (b - a > 1) {
        const long long m = (a + b) >> 1;
        if (seg_off[m] <= jj) a = m; else b = m;
      }
      src = utt_off[a] + sb;
    }
    long long tot, tot_z;
    long long x = len;
    speech_block_scan2<kSpeechThreads>(x, zero, sh_sum, tot, tot_z);
    s_dst[threadIdx.x] = dst + x;
    s_src[threadIdx.x] = src - (dst + x);
    if (threadIdx.x == 0) s_dst[kSpeechThreads] = dst + tot;
    __syncthreads();
    const long long b0 = dst > lo ? dst : lo, b1 = dst + tot < hi_s ? dst + tot : hi_s;
    // vectors of 8 samples in [b0, b1): b0 is a multiple of 8; the last one may be cut by out_capacity
    const long long v0 = b0 >> 3, v1 = (b1 + 7) >> 3;
    for (long long v = v0 + threadIdx.x; v < v1; v += kSpeechThreads * kGatherUnroll) {
      int4 val[kGatherUnroll];
      long long o[kGatherUnroll];
      const int16_t* src_p[kGatherUnroll];
#pragma unroll
      for (int q = 0; q < kGatherUnroll; ++q) {
        const long long vv = v + static_cast<long long>(q) * kSpeechThreads;
        o[q] = vv << 3;
        if (vv < v1) {
          int lo_i = 0, hi_i = kSpeechThreads;  // batch segment k with s_dst[k] <= o < s_dst[k + 1]
          while (hi_i - lo_i > 1) {
            const int m = (lo_i + hi_i) >> 1;
            if (s_dst[m] <= o[q]) lo_i = m; else hi_i = m;
          }
          src_p[q] = pcm + s_src[lo_i] + o[q];
          val[q] = __ldg(reinterpret_cast<const int4*>(src_p[q]));
        }
      }
#pragma unroll
      for (int q = 0; q < kGatherUnroll; ++q) {
        const long long vv = v + static_cast<long long>(q) * kSpeechThreads;
        if (vv >= v1) continue;
        if (o[q] + 8 <= b1) {
          *reinterpret_cast<int4*>(out + o[q]) = val[q];
        } else {
          for (int k = 0; o[q] + k < b1; ++k) out[o[q] + k] = src_p[q][k];  // cut by out_capacity
        }
      }
    }
    dst += tot;
    j += kSpeechThreads;
    __syncthreads();
  }
}

// Stream bank: end the streams with end[s] != 0.  One thread per stream: with speech on (g.meta != nullptr) it
// drains the stream's pending rows in shared memory (its rings, lane-strided) and writes the tail; then it zeroes
// the stream's bank state (history [n][320], MFCC ring [65][n], fed, previous sample) so its next chunk starts a
// new signal.  Shared memory: (W1 + W2) * kSegEndThreads words.
__global__ void __launch_bounds__(kSegEndThreads) stream_end_kernel(
    const StreamSeg g, const uint8_t* __restrict__ end, int n_streams, int16_t* __restrict__ hist,
    float* __restrict__ mfcc_ring, int* __restrict__ fed, int16_t* __restrict__ prev, uint8_t* __restrict__ tail_rows,
    int64_t* __restrict__ tail_bounds) {
  extern __shared__ uint32_t seg_scratch[];
  const int s = blockIdx.x * kSegEndThreads + threadIdx.x;
  if (s >= n_streams || !end[s]) return;
  const int f = fed[s];
  if (g.meta) seg_end(g, s, f > 7 ? f - 7 : 0, seg_scratch + threadIdx.x, kSegEndThreads, tail_rows, tail_bounds);
  uint32_t* h32 = reinterpret_cast<uint32_t*>(hist + static_cast<long long>(s) * 320);
  for (int k = 0; k < 160; ++k) h32[k] = 0;
  for (int k = 0; k < 65; ++k) mfcc_ring[static_cast<long long>(k) * n_streams + s] = 0.0f;
  fed[s] = 0;
  prev[s] = 0;
}

// Ragged bank: the same for the streams with end[s] != 0, with R the rows the stream has emitted (vad_ragged.h
// ragged_rows of its sample count N).  Then N and the MFCC ring are zero: samples that have not completed a frame are
// discarded, and the sample ring needs no clearing (a new signal's frames read only its own samples).
__global__ void __launch_bounds__(kSegEndThreads) stream_end_ragged_kernel(
    const StreamSeg g, const uint8_t* __restrict__ end, int n_streams, long long* __restrict__ total,
    float* __restrict__ mfcc_ring, uint8_t* __restrict__ tail_rows, int64_t* __restrict__ tail_bounds) {
  extern __shared__ uint32_t seg_scratch[];
  const int s = blockIdx.x * kSegEndThreads + threadIdx.x;
  if (s >= n_streams || !end[s]) return;
  if (g.meta)
    seg_end(g, s, static_cast<int>(ragged_rows(total[s])), seg_scratch + threadIdx.x, kSegEndThreads, tail_rows,
            tail_bounds);
  for (int k = 0; k < 65; ++k) mfcc_ring[static_cast<long long>(k) * n_streams + s] = 0.0f;
  total[s] = 0;
}

#endif  // __CUDACC__

}  // namespace vadb
