// Host emulation of the stream bank's online speech segments (vad_segments.cuh seg_step / seg_end, run by
// stream_feed_speech_kernel and stream_end_kernel) -- TEST INFRASTRUCTURE.  Keeps the kernels' state layout:
// struct-of-arrays over streams with the same ring words, and the end kernel's lane-strided scratch per block of
// kSegEndThreads streams.  The product never links this file.
#include <cstdint>
#include <vector>

#include "../../vad_b200/csrc/vad_segments.cuh"

using namespace vadb;

namespace {

struct EmulBank {
  int n;
  std::vector<int> fed;
  std::vector<uint32_t> seg;  // [W1 + W2 + 2][n], as vadb200_stream_bank_set_speech allocates it
  StreamSeg g;
};

}  // namespace

extern "C" {

// A bank of n streams with speech on at (S, G, P); nullptr on a bad argument.
void* emul_bank_create(int n, int min_speech_rows, int min_silence_rows, int pad_rows) {
  if (n < 1) return nullptr;
  for (int v : {min_speech_rows, min_silence_rows, pad_rows})
    if (v < 0 || v > kSpeechMaxParam) return nullptr;
  EmulBank* b = new EmulBank();
  b->n = n;
  b->fed.assign(n, 0);
  const SmoothParams sp = smooth_params(min_speech_rows, min_silence_rows, pad_rows);
  StreamSeg& g = b->g;
  g = StreamSeg{};
  g.n = n;
  g.G = sp.G; g.S = sp.S; g.P = sp.P; g.H = sp.H;
  g.d1 = sp.G > 1 ? sp.G - 1 : 0;
  g.d2 = sp.S > 1 ? sp.S - 1 : 0;
  const long long w1 = g.d1 ? seg_ring_words(g.d1) : 0, w2 = g.d2 ? seg_ring_words(g.d2) : 0;
  b->seg.assign(static_cast<size_t>(w1 + w2 + 2) * n, 0u);
  g.ring1 = b->seg.data();
  g.ring2 = b->seg.data() + w1 * n;
  g.meta = b->seg.data() + (w1 + w2) * n;
  g.last = reinterpret_cast<int*>(g.meta + n);
  return b;
}

void emul_bank_destroy(void* p) { delete static_cast<EmulBank*>(p); }

int emul_bank_delay(void* p) { return static_cast<EmulBank*>(p)->g.H; }

// State words per stream (rings, meta, last).
long long emul_bank_state_words(void* p) {
  const EmulBank* b = static_cast<EmulBank*>(p);
  return static_cast<long long>(b->seg.size()) / b->n;
}

// One tick: decisions[i] is stream i's FFN decision (0 / 1).  As the feed kernel does, the label is 255 while the
// stream has fed fewer than 7 chunks; otherwise it is row fed - 7.  Writes labels, rows and bounds [n].
void emul_bank_feed(void* p, const uint8_t* decisions, uint8_t* labels, uint8_t* rows, int64_t* bounds) {
  EmulBank* b = static_cast<EmulBank*>(p);
  for (int s = 0; s < b->n; ++s) {
    const int fedl = b->fed[s];
    const uint8_t lab = fedl - 2 >= 5 ? decisions[s] : 255;
    b->fed[s] = fedl + 1;
    uint8_t row = 255;
    long long bound = -1;
    if (lab != 255) seg_step(b->g, s, fedl - 7, lab != 0, row, bound);
    labels[s] = lab;
    rows[s] = row;
    bounds[s] = bound;
  }
}

// stream_end_kernel over blocks of kSegEndThreads streams, each block with its own lane-strided scratch.
void emul_bank_end(void* p, const uint8_t* end, uint8_t* tail_rows, int64_t* tail_bounds) {
  EmulBank* b = static_cast<EmulBank*>(p);
  const StreamSeg& g = b->g;
  const int words = (g.d1 ? seg_ring_words(g.d1) : 0) + (g.d2 ? seg_ring_words(g.d2) : 0);
  std::vector<uint32_t> scratch(static_cast<size_t>(words) * kSegEndThreads + 1, 0xdeadbeefu);
  for (int s = 0; s < b->n; ++s) {
    if (!end[s]) continue;
    const int f = b->fed[s];
    seg_end(g, s, f > 7 ? f - 7 : 0, scratch.data() + s % kSegEndThreads, kSegEndThreads, tail_rows, tail_bounds);
    b->fed[s] = 0;
  }
}

}  // extern "C"
