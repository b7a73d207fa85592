// Host emulation of the ragged stream bank's sample ring (vad_ragged.h, as stream_ragged_kernel uses it) -- TEST
// INFRASTRUCTURE.  One stream: each feed appends its packet to the ring from slot N mod R on, then stages every frame
// the packet completes the way the kernel does (its first word, 200 words stepping with ragged_wrap, the sample
// before it), and advances the first word by 80 per frame.  The product never links this file.
#include <cstdint>
#include <vector>

#include "../../vad_b200/csrc/vad_ragged.h"

using namespace vadb;

extern "C" {

// Feed packets of sizes[0 .. n_feeds) (consecutive pieces of `signal`) to one stream of a bank with cap `cap`.  For
// every frame staged, in order: frame[k] its index, staged[k][401] the sample before it then its 400 samples,
// row[k] the row it emits (-1: none) and slot[k] that row's output slot in its feed (-1: none).  counts[t] gets the
// rows feed t emits.  Returns the frames staged; -1 when a size is outside [0, cap] or there are more than
// max_frames.  Unwritten ring slots hold 0x7777, so a read of one shows in the staged samples.
long long emul_ragged_stream(int cap, int n_feeds, const int* sizes, const int16_t* signal, long long max_frames,
                             long long* frame, int16_t* staged, long long* row, int* slot, int* counts) {
  const int R = ragged_ring_samples(cap), K = ragged_max_rows(cap);
  if (R % 160 != 0 || R < cap + 401) return -1;
  std::vector<int16_t> ring(R, 0x7777);
  long long N = 0, pos = 0, k = 0;
  for (int t = 0; t < n_feeds; ++t) {
    const int c = sizes[t];
    if (c < 0 || c > cap) return -1;
    const long long f0 = ragged_frames(N);
    const int nf = static_cast<int>(ragged_frames(N + c) - f0);
    const int cnt = static_cast<int>(ragged_rows(N + c) - ragged_rows(N));
    if (cnt > K) return -1;
    const int base = ragged_slot(N, R);
    int w0 = ragged_frame_word0(f0, R);
    for (int q = 0; q < c; ++q) ring[ragged_wrap(base + q, R)] = signal[pos + q];
    for (int j = 0; j < nf; ++j) {
      if (k >= max_frames) return -1;
      const long long f = f0 + j;
      int16_t* out = staged + 401 * k;
      out[0] = f > 0 ? ring[ragged_pre_slot(w0, R)] : 0;
      for (int wd = 0; wd < 200; ++wd) {
        const int x = ragged_wrap(w0 + wd, R / 2);
        out[1 + 2 * wd] = ring[2 * x];
        out[2 + 2 * wd] = ring[2 * x + 1];
      }
      w0 = ragged_wrap(w0 + 80, R / 2);
      frame[k] = f;
      row[k] = f >= 5 ? f - 5 : -1;
      slot[k] = f >= 5 ? static_cast<int>(f - (f0 > 5 ? f0 : 5)) : -1;
      ++k;
    }
    counts[t] = cnt;
    N += c;
    pos += c;
  }
  return k;
}

int emul_ragged_max_rows(int cap) { return ragged_max_rows(cap); }
int emul_ragged_ring_samples(int cap) { return ragged_ring_samples(cap); }

}  // extern "C"
