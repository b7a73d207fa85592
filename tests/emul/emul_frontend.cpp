// Host emulation of the front-end variant (fused_fe_kernel, frames_kernel with a front end) -- TEST INFRASTRUCTURE.
// Builds on emul.cpp (same translation unit: its tables, thread model and exchange loops) and swaps the per-thread
// loads for vad_core.cuh's fft_load_pcm2_fe / fft_load_f32_fe, staging each step the way the kernel does: 8 samples
// into the buffer, the sample before the step just below it (0 at the utterance start), so the previous-sample
// reads (word m - 1, word -1 for the step's first frame) run through the same index math.
// The product never links this file.
#include "emul.cpp"

namespace {

struct FrontEndEmul {
  float preemph;
  cf2 win[kFftN / 2];  // window pairs, ones past sample 400 (the handle's device table)
};

FrontEndEmul make_fe(float preemph, const float* window) {
  FrontEndEmul fe;
  fe.preemph = preemph;
  for (int m = 0; m < kFftN / 2; ++m)
    fe.win[m] = (window && m < kFrame / 2) ? cf2{window[2 * m], window[2 * m + 1]} : cf2{1.0f, 1.0f};
  return fe;
}

// warp_fft_quad for one half-warp with the front-end load (see fft_pair_pcm in emul.cpp)
void fft_pair_pcm_fe(const uint32_t* w32a, int delta, float* P2, int col, const FrontEndEmul& fe) {
  PairThreads th;
  std::vector<f2> ex(kExchFrame);
  for (int t = 0; t < 16; ++t) {
    fft_load_pcm2_fe(w32a, delta, t, fe.preemph, fe.win, th.xr[t], th.xi[t]);
    fft_pass1<13>(th.xr[t], th.xi[t], g_tw1, t);
  }
  for (int t = 0; t < 16; ++t) exch_store_plane(ex.data(), t, th.xr[t]);
  for (int k1 = 0; k1 < 16; ++k1) exch_load_plane(ex.data(), k1, th.xr[k1]);
  for (int t = 0; t < 16; ++t) exch_store_plane(ex.data(), t, th.xi[t]);
  for (int k1 = 0; k1 < 16; ++k1) exch_load_plane(ex.data(), k1, th.xi[k1]);
  for (int k1 = 0; k1 < 16; ++k1) dft16<16>(th.xr[k1], th.xi[k1]);
  static f2 sr[16][16], si[16][16];
  for (int k1 = 0; k1 < 16; ++k1)
    for (int j = 8; j < 16; ++j) {
      sr[k1][j] = (k1 == 0) ? th.xr[k1][(j + 1) & 15] : th.xr[k1][j];
      si[k1][j] = (k1 == 0) ? th.xi[k1][(j + 1) & 15] : th.xi[k1][j];
    }
  for (int k1 = 0; k1 < 16; ++k1) {
    auto xch = [&](f2, int j, bool imag, int partner) { return imag ? si[partner][j] : sr[partner][j]; };
    auto store = [&](int bin, f2 v) {
      if (bin >= kMelFirstBin) {
        P2[p2_index(bin, col)] = v.x;
        P2[p2_index(bin, col) + 2] = v.y;
      }
    };
    fft_split_store(th.xr[k1], th.xi[k1], k1, g_tw2, xch, store);
  }
}

void fft_frame_f32_fe(const float* fr, int frame_len, float* Pcol, const FrontEndEmul& fe) {
  FrameThreads th;
  std::vector<cf2> ex(kExchFrame);
  for (int t = 0; t < 16; ++t) {
    fft_load_f32_fe(fr, frame_len, t, fe.preemph, fe.win, th.xr[t], th.xi[t]);
    fft_pass1<16>(th.xr[t], th.xi[t], g_tw1, t);
    exch_store(ex.data(), t, th.xr[t], th.xi[t]);
  }
  for (int k1 = 0; k1 < 16; ++k1) {
    exch_load(ex.data(), k1, th.xr[k1], th.xi[k1]);
    dft16<16>(th.xr[k1], th.xi[k1]);
  }
  float sr[16][16], si[16][16];
  for (int k1 = 0; k1 < 16; ++k1)
    for (int j = 8; j < 16; ++j) {
      sr[k1][j] = (k1 == 0) ? th.xr[k1][(j + 1) & 15] : th.xr[k1][j];
      si[k1][j] = (k1 == 0) ? th.xi[k1][(j + 1) & 15] : th.xi[k1][j];
    }
  for (int k1 = 0; k1 < 16; ++k1) {
    auto xch = [&](float, int j, bool imag, int partner) { return imag ? si[partner][j] : sr[partner][j]; };
    auto store = [&](int bin, float v) { Pcol[bin * kPPitch] = v; };
    fft_split_store(th.xr[k1], th.xi[k1], k1, g_tw2, xch, store);
  }
}

}  // namespace

extern "C" {

// emul_spec_f32 with the front end (window: 400 weights or null); each frame is its own signal
int emul_spec_f32_fe(const float* frames, int n_frames, int frame_len, float preemph, const float* window,
                     float* spec /*[n][256]*/) {
  if (!g_init) return -1;
  const FrontEndEmul fe = make_fe(preemph, window);
  std::vector<float> P(256 * kPPitch);
  for (int f = 0; f < n_frames; ++f) {
    fft_frame_f32_fe(frames + static_cast<size_t>(f) * frame_len, frame_len, P.data(), fe);
    for (int k = 0; k < 256; ++k) spec[static_cast<size_t>(f) * 256 + k] = P[k * kPPitch] * 9.5367431640625e-07f;
  }
  return 0;
}

// emul_utterance through the front-end variant: pre-emphasis + window (400 weights or null) and the decision
// threshold (<= 0: argmax).  Outputs as emul_utterance (any may be null).
int emul_utterance_fe(const int16_t* pcm, long long n_samples, int feat_mode, float preemph, const float* window,
                      float thresh, float* mfcc_out, float* feats_out, float* logits_out, uint8_t* labels_out) {
  if (!g_init) return -1;
  const FrontEndEmul fe = make_fe(preemph, window);
  const long long T = frames_for_length(n_samples);
  if (T <= 0) return 0;
  const int n = static_cast<int>(T);
  const int nsteps = (n + kStepFrames - 1) / kStepFrames;
  std::vector<float> P(kP2RowsAlloc * kP2Pitch), logE(kNMel * 32), ring(kNCep * kRing);
  std::vector<int16_t> stage_buf(kStageSamples + 16);
  int out_done = 2;
  for (int s = 0; s < nsteps; ++s) {
    const long long start = static_cast<long long>(s) * kStepFrames * kHop;
    const long long avail = std::min<long long>(n_samples - start, kStageSamples);
    std::memset(stage_buf.data(), 0x55, stage_buf.size() * sizeof(int16_t));  // stale garbage around the data
    int16_t* stage = stage_buf.data() + 8;
    std::memcpy(stage, pcm + start, static_cast<size_t>(avail) * sizeof(int16_t));
    stage[-1] = s > 0 ? pcm[start - 1] : int16_t(0);
    for (int w = 0; w < 8; ++w)
      for (int h = 0; h < 2; ++h) {
        const uint32_t* w32 = reinterpret_cast<const uint32_t*>(stage) + (4 * w + h) * (kHop / 2);
        fft_pair_pcm_fe(w32, kHop, P.data(), col_of_halfwarp(w, h), fe);
      }
    for (int g = 0; g < 8; ++g)
      for (int lane = 0; lane < 32; ++lane) mel2_run_dispatch<kP2Pitch, 32>(g, P.data() + 2 * lane, logE.data() + lane);
    for (int w = 0; w < 7; ++w)
      for (int lane = 0; lane < 32; ++lane) {
        const int f = s * kStepFrames + slot_of_col(lane);
        float ra, rb;
        dct_coef2<32>(logE.data() + lane, w, ra, rb);
        ring[2 * w * kRing + f % kRing] = ra;
        if (2 * w + 1 < kNCep) ring[(2 * w + 1) * kRing + f % kRing] = rb;
      }
    const int computed = std::min((s + 1) * kStepFrames, n);
    if (mfcc_out)
      for (int f = s * kStepFrames; f < computed; ++f)
        for (int c = 0; c < kNCep; ++c) mfcc_out[static_cast<size_t>(f) * kNCep + c] = ring[c * kRing + f % kRing];
    if (((s + 1) & 7) == 0 || s == nsteps - 1) {
      const int last_center = std::min(computed - 3, n - 4);
      for (int c = out_done; c <= last_center; ++c) {
        float r[5][kNCep];
        for (int d = 0; d < 5; ++d)
          for (int k = 0; k < kNCep; ++k) r[d][k] = ring[k * kRing + (c - 2 + d) % kRing];
        float x[kNFeat];
        const bool ok = window_features(r, feat_mode, x);
        float logit[kNCls];
        ffn_forward(g_ffn, x, logit);
        uint8_t lab = decide(logit, thresh);
        if (!ok) { logit[0] = logit[1] = logit[2] = NAN; lab = 0; }
        const size_t row = static_cast<size_t>(c - 2);
        if (feats_out) std::memcpy(feats_out + row * kNFeat, x, sizeof(x));
        if (logits_out) std::memcpy(logits_out + row * kNCls, logit, sizeof(logit));
        if (labels_out) labels_out[row] = lab;
      }
      out_done = std::max(out_done, last_center + 1);
    }
  }
  return 0;
}

}  // extern "C"

// ---- float32 power spectra and tables for the spectrum -> MFCC bound (tests/_mfcc_bound.py) ----------------------------
extern "C" {

// Raw |2X|^2 of every frame of one utterance through the fused kernel's load path: fft_load_pcm2 (use_fe == 0) or
// fft_load_pcm2_fe (previous sample 0 at the utterance start), pass 1 with NZ = 13, the pair tile and
// fft_split_store.  out [T][256]: bins kMelFirstBin .. 255 (bin 128 from thread 0's self-paired store); the bins the
// kernel drops stay NaN, and so does any bin no store reached.
int emul_power_pcm(const int16_t* pcm, long long n_samples, int use_fe, float preemph, const float* window,
                   float* out) {
  if (!g_init) return -1;
  const FrontEndEmul fe = make_fe(preemph, window);
  const long long T = frames_for_length(n_samples);
  const int n = static_cast<int>(T);
  const int nsteps = (n + kStepFrames - 1) / kStepFrames;
  std::vector<float> P(kP2RowsAlloc * kP2Pitch);
  std::vector<int16_t> stage_buf(kStageSamples + 16);
  for (int s = 0; s < nsteps; ++s) {
    const long long start = static_cast<long long>(s) * kStepFrames * kHop;
    const long long avail = std::min<long long>(n_samples - start, kStageSamples);
    std::memset(stage_buf.data(), 0x55, stage_buf.size() * sizeof(int16_t));
    int16_t* stage = stage_buf.data() + 8;
    std::memcpy(stage, pcm + start, static_cast<size_t>(avail) * sizeof(int16_t));
    stage[-1] = s > 0 ? pcm[start - 1] : int16_t(0);
    std::fill(P.begin(), P.end(), NAN);
    for (int w = 0; w < 8; ++w)
      for (int h = 0; h < 2; ++h) {
        const uint32_t* w32 = reinterpret_cast<const uint32_t*>(stage) + (4 * w + h) * (kHop / 2);
        if (use_fe) fft_pair_pcm_fe(w32, kHop, P.data(), col_of_halfwarp(w, h), fe);
        else fft_pair_pcm(w32, kHop, P.data(), col_of_halfwarp(w, h));
      }
    for (int col = 0; col < kStepFrames; ++col) {
      const long long f = static_cast<long long>(s) * kStepFrames + slot_of_col(col);
      if (f >= n) continue;
      for (int k = 0; k < kBins; ++k)
        out[f * kBins + k] = k >= kMelFirstBin ? P[p2_index(k, col)] : NAN;
    }
  }
  return 0;
}

// Raw |2X|^2 [n][256] of explicit float frames through frames_kernel's path: fft_load_f32 (use_fe == 0) or
// fft_load_f32_fe, pass 1 with NZ = 16, one frame per thread.  get_spec_mag is this times 2^-20.
int emul_power_f32(const float* frames, int n_frames, int frame_len, int use_fe, float preemph, const float* window,
                   float* out) {
  if (!g_init) return -1;
  const FrontEndEmul fe = make_fe(preemph, window);
  std::vector<float> P(256 * kPPitch);
  for (int f = 0; f < n_frames; ++f) {
    const float* fr = frames + static_cast<size_t>(f) * frame_len;
    std::fill(P.begin(), P.end(), NAN);
    if (use_fe) fft_frame_f32_fe(fr, frame_len, P.data(), fe);
    else fft_frame_f32(fr, frame_len, P.data());
    for (int k = 0; k < 256; ++k) out[static_cast<size_t>(f) * 256 + k] = P[k * kPPitch];
  }
  return 0;
}

// The float32 tables the kernels read, as dense matrices: melw (mel_group: frames_kernel, spec_to_mfcc_kernel) and
// melw2 (mel2_run: the fused kernels) [26][256], both x 2^-20; dct (dct_coef) and dctp (dct_coef2 / dct_coef4)
// [13][26].
int emul_tables(float* melw, float* melw2, float* dct, float* dctp) {
  if (!g_init) return -1;
  std::memset(melw, 0, kNMel * kBins * sizeof(float));
  std::memset(melw2, 0, kNMel * kBins * sizeof(float));
  for (int m = 0; m < kNMel; ++m) {
    for (int k = kMelLo[m]; k < kMelHi[m]; ++k) melw[m * kBins + k] = c_tab.melw[kMelOff[m] + k - kMelLo[m]];
    for (int q = 0; q < mel_nq(m); ++q)
      for (int e = 0; e < 2; ++e) melw2[m * kBins + 2 * (mel_q0(m) + q) + e] = c_tab.melw2[2 * (mel_qoff(m) + q) + e];
  }
  std::memcpy(dct, c_tab.dct, kNCep * kNMel * sizeof(float));
  for (int k = 0; k < kNCep; ++k)
    for (int n = 0; n < kNMel; ++n) dctp[k * kNMel + n] = c_tab.dctp[k >> 1][n][k & 1];
  return 0;
}

// Read (set == 0) or replace (set != 0) the FFT twiddle tables tw1 [256] and tw2 [128] as (re, im) pairs: the CPU
// suite's mutants of the replay.  emul_init restores the host's own tables.
int emul_twiddles(float* tw1, float* tw2, int set) {
  if (!g_init) return -1;
  if (set) {
    std::memcpy(g_tw1, tw1, sizeof(g_tw1));
    std::memcpy(g_tw2, tw2, sizeof(g_tw2));
  } else {
    std::memcpy(tw1, g_tw1, sizeof(g_tw1));
    std::memcpy(tw2, g_tw2, sizeof(g_tw2));
  }
  return 0;
}

}  // extern "C"
