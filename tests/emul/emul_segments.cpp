// Host emulation of the speech-segment smoothing kernel (vad_segments.cuh speech_smooth_kernel) -- TEST
// INFRASTRUCTURE.  Drives the kernel's own __host__ __device__ tile functions through its tile, window and chunk
// index math: tiles of kSpeechTile rows per utterance, windows with the H-row halo, one chunk per thread, and the
// block-wide edge scans done serially.  The product never links this file.
#include <algorithm>
#include <cstdint>
#include <vector>

#include "../../vad_b200/csrc/vad_segments.cuh"

using namespace vadb;

extern "C" {

// labels [rows] of n_utt utterances with row offsets row_off [n_utt + 1]; tile = rows per tile (kSpeechTile in the
// product, smaller here to put many tile edges in a short test).  Writes smoothed [rows]; returns the number of
// segment starts or -1 on a bad argument.
long long emul_speech_smooth(const uint8_t* labels, const long long* row_off, long long n_utt, int min_speech_rows,
                             int min_silence_rows, int pad_rows, int tile, uint8_t* smoothed) {
  if (tile < 1 || tile > kSpeechTile) return -1;
  const SmoothParams sp = smooth_params(min_speech_rows, min_silence_rows, pad_rows);
  const int cap = (smooth_window_cap(sp.H) + 15) & ~15;
  std::vector<uint8_t> a(cap), b(cap);
  std::vector<int16_t> prv(cap);
  std::vector<int> last(kSpeechThreads), first(kSpeechThreads), lin(kSpeechThreads), rin(kSpeechThreads);
  std::vector<int> c0(kSpeechThreads), c1(kSpeechThreads);
  long long starts = 0;
  auto scan = [&](int n) {  // speech_block_edges
    int run = -1;
    for (int t = 0; t < kSpeechThreads; ++t) {
      lin[t] = run;
      run = run > last[t] ? run : last[t];
    }
    run = n;
    for (int t = kSpeechThreads - 1; t >= 0; --t) {
      rin[t] = run;
      run = run < first[t] ? run : first[t];
    }
  };
  for (long long u = 0; u < n_utt; ++u) {
    const long long ubeg = row_off[u], uend = row_off[u + 1];
    for (long long r0 = ubeg; r0 < uend; r0 += tile) {
      SpeechTile t{r0, static_cast<int>(uend - r0 < tile ? uend - r0 : tile), static_cast<int>(u)};
      const SmoothWindow w = smooth_window(t, ubeg, uend, sp.H);
      if (w.n > cap) return -1;
      std::fill(a.begin(), a.end(), 0xAA);  // rows no step writes stay visibly foreign
      std::fill(b.begin(), b.end(), 0xAA);
      for (int tid = 0; tid < kSpeechThreads; ++tid) {
        smooth_chunk(w.n, tid, c0[tid], c1[tid]);
        smooth_load(labels, w.w0, w.n, c0[tid], c1[tid], a.data(), last[tid], first[tid]);
      }
      scan(w.n);
      for (int tid = 0; tid < kSpeechThreads; ++tid) {
        smooth_fill(a.data(), b.data(), prv.data(), w.n, c0[tid], c1[tid], lin[tid], rin[tid], sp.G);
        smooth_edges(b.data(), w.n, c0[tid], c1[tid], 0, last[tid], first[tid]);
      }
      scan(w.n);
      for (int tid = 0; tid < kSpeechThreads; ++tid) {
        smooth_runs(b.data(), a.data(), prv.data(), c0[tid], c1[tid], lin[tid], rin[tid], sp.S);
        smooth_edges(a.data(), w.n, c0[tid], c1[tid], 1, last[tid], first[tid]);
      }
      scan(w.n);
      for (int tid = 0; tid < kSpeechThreads; ++tid)
        smooth_pad(a.data(), b.data(), prv.data(), w.n, c0[tid], c1[tid], lin[tid], rin[tid], sp.P, w.o0, w.o1);
      for (int i = w.t0; i < w.o1; ++i) {
        smoothed[w.w0 + i] = b[i];
        starts += seg_starts(b.data(), w.o0, i);
      }
    }
  }
  return starts;
}

int emul_speech_window(long long r0, int n, long long ubeg, long long uend, int H, long long* out /* w0 n o0 t0 o1 */) {
  const SmoothWindow w = smooth_window(SpeechTile{r0, n, 0}, ubeg, uend, H);
  out[0] = w.w0; out[1] = w.n; out[2] = w.o0; out[3] = w.t0; out[4] = w.o1;
  return 0;
}

}  // extern "C"
