// vad_ragged.h -- index math of the ragged stream bank (vadb200_stream_bank_create_ragged): which frames a feed
// completes, which row each one emits, and where a frame's samples sit in the stream's sample ring.  Plain C++ marked
// __host__ __device__: stream_ragged_kernel and stream_end_ragged_kernel use it, and tests/emul/emul_stream_ragged.cpp
// drives the same functions on the host.
//
// A stream that has taken N samples since its last reset or end has completed the frames f >= 0 with
// 160 f + 400 <= N.  Completing frame f >= 5 emits row f - 5 (it classifies frame f - 3 from the MFCC ring holding
// frames f - 5 .. f - 1: the fixed bank's "chunk r + 7 emits row r").  The stream's last R samples live in a ring of
// R = ragged_ring_samples(cap) int16 (sample i at slot i mod R); R is a multiple of 160, so every frame starts on a
// 32-bit word, and R >= cap + 401 holds a whole feed plus the oldest frame it can still complete and the sample
// before that frame (pre-emphasis).
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define VADB_RAG_HD __host__ __device__ __forceinline__
#else
#define VADB_RAG_HD inline
#endif

namespace vadb {

constexpr int kRaggedMaxFeed = 16000;  // samples one stream may take in one feed (1 s)

// Frames completed by n samples.
VADB_RAG_HD long long ragged_frames(long long n) { return n >= 400 ? (n - 400) / 160 + 1 : 0; }
// Rows emitted by n samples (= the rows of an offline utterance of n + 1 samples).
VADB_RAG_HD long long ragged_rows(long long n) {
  const long long f = ragged_frames(n);
  return f > 5 ? f - 5 : 0;
}
// K: the most rows one feed of at most cap samples can emit.
VADB_RAG_HD int ragged_max_rows(int cap) { return (cap + 159) / 160; }
// R: samples in each stream's ring.
VADB_RAG_HD int ragged_ring_samples(int cap) { return 160 * ((cap + 401 + 159) / 160); }
// Ring slot of sample i (one 64-bit remainder per stream and feed; the kernels step from there with ragged_wrap).
VADB_RAG_HD int ragged_slot(long long i, int R) { return static_cast<int>(i % R); }
// x mod m for 0 <= x < 2 m: a slot (or word) plus an offset below the ring's length.
VADB_RAG_HD int ragged_wrap(int x, int m) { return x >= m ? x - m : x; }
// Ring word of frame f's first two samples; frame f + 1 starts 80 words later (mod R / 2).  Word w < 200 of the
// frame is ragged_wrap(w0 + w, R / 2): a frame may wrap the ring.
VADB_RAG_HD int ragged_frame_word0(long long f, int R) { return ragged_slot(160 * f, R) / 2; }
// Ring slot of the sample before the frame that starts at word w0 (pre-emphasis; frame 0 takes 0 instead).
VADB_RAG_HD int ragged_pre_slot(int w0, int R) { return w0 > 0 ? 2 * w0 - 1 : R - 1; }

}  // namespace vadb
