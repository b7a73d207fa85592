// Host emulation of the resampling ragged bank's source-rate side (vad_stream_resample.h, as the plan step and
// stream_resample_kernel use it) -- TEST INFRASTRUCTURE.  One stream: each feed computes its output count and tiles,
// stages every tile's window from the history and the packet, runs the polyphase sum in float64 and writes the new
// history from the last tile's window, double-buffered as on the device.  The product never links this file.
#include <cstdint>
#include <vector>

#include "../../vad_b200/csrc/vad_stream_resample.h"

using namespace vadb;

extern "C" {

long long emul_srs_ready(long long n, int up, int down, int half) { return srs_ready(n, up, down, half); }
int emul_srs_cap16(int cap, int up, int down) { return srs_cap16(cap, up, down); }
int emul_srs_window_max(int up, int down, int K) { return srs_window_max(up, down, K); }

// Feed packets of sizes[0 .. n_feeds) (consecutive pieces of `signal`) to one stream with packet cap `cap`.  poly is
// the polyphase table [up][K] (row p: h[p], h[p + up], ...; zeros past the filter), in float64.  out gets every
// output in order; counts[t] / tiles[t] the outputs and tiles of feed t; *widest the largest window staged.  Returns
// the outputs, or -1 when a size is outside [0, cap], a feed adds more than cap16 outputs, a window exceeds
// srs_window_max, or a window or history index leaves its buffer.
long long emul_srs_stream(int up, int down, int half, int K, int cap, int n_feeds, const int* sizes,
                          const int16_t* signal, const double* poly, double* out, int* counts, int* tiles,
                          int* widest) {
  const int hs = K - 1, cap16 = srs_cap16(cap, up, down), wmax = srs_window_max(up, down, K);
  std::vector<int16_t> hist[2] = {std::vector<int16_t>(hs, 0), std::vector<int16_t>(hs, 0)};
  std::vector<double> win;
  int cur = 0;
  long long N = 0, pos = 0, n_out = 0;
  *widest = 0;
  for (int t = 0; t < n_feeds; ++t) {
    const int c = sizes[t];
    if (c < 0 || c > cap) return -1;
    const long long m0 = srs_ready(N, up, down, half);
    const int outs = static_cast<int>(srs_ready(N + c, up, down, half) - m0);
    if (outs > cap16) return -1;
    const int nt = srs_tiles(c, outs);
    counts[t] = outs;
    tiles[t] = nt;
    const int rd = cur;
    for (int j = 0; j < nt; ++j) {
      const long long ma = m0 + static_cast<long long>(j) * kSrsTile;
      const long long mb = ma + kSrsTile < m0 + outs ? ma + kSrsTile : m0 + outs;
      const bool last = j == nt - 1;
      const SrsWindow w = srs_window(ma, mb, last, N + c, up, down, half, K);
      const long long nw = w.hi - w.lo + 1;
      if (nw > wmax || nw < 0) return -1;
      if (nw > *widest) *widest = static_cast<int>(nw);
      win.assign(nw, 0.0);
      for (long long k = 0; k < nw; ++k) {
        const long long g = w.lo + k;
        if (g < N) {
          const int s = srs_hist_slot(g, N, K);
          if (s < 0 || s >= hs) return -1;
          win[k] = hist[rd][s];
        } else {
          if (g - N >= c) return -1;
          win[k] = signal[pos + (g - N)];
        }
      }
      for (long long m = ma; m < mb; ++m) {
        const long long tt = m * down + half;
        const long long z = tt / up - w.lo;
        if (z - (K - 1) < 0 || z >= nw) return -1;
        const double* hr = poly + (tt % up) * K;
        double acc = 0.0;
        for (int i = 0; i < K; ++i) acc += hr[i] * win[z - i];
        out[n_out + (m - m0)] = acc;
      }
      if (last) {
        const long long k0 = N + c - (K - 1) - w.lo;
        if (k0 < 0 || k0 + hs > nw) return -1;
        for (int k = 0; k < hs; ++k) hist[rd ^ 1][k] = static_cast<int16_t>(win[k0 + k]);
      }
    }
    if (c > 0) cur ^= 1;
    n_out += outs;
    N += c;
    pos += c;
  }
  return n_out;
}

}  // extern "C"
