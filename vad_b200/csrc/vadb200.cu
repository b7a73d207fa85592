// vadb200.cu -- C ABI (include/vadb200.h) over the sm_100a kernels of vad_kernels.cuh.
// Host logic only: handle / plan / bank lifetime, segment tables, launches, the chunked
// H2D -> kernel -> D2H pipeline of vadb200_vad_host.  No CPU compute path exists: every
// numeric entry point launches a CUDA kernel or fails with VADB200_E_CUDA.
#include "../../include/vadb200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "vad_host_tables.h"
#include "vad_kernels.cuh"
#include "ffn_train.cuh"
#include "vad_segments.cuh"
#include "vad_resample.cuh"

using namespace vadb;

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};
std::atomic<unsigned long long> g_next_id{1};
std::mutex g_tab_mu;
bool g_tab_loaded[64] = {false};  // per device: mel / DCT tables uploaded (config-invariant content)

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return VADB200_E_CUDA;
}
#define CU(expr)                                     \
  do {                                               \
    cudaError_t e__ = (expr);                        \
    if (e__ != cudaSuccess) return cuda_fail(e__, #expr); \
  } while (0)

// Every kernel launch goes through here: `enqueue` launches n kernels.  The thread's last error is cleared first, so
// the check reports these launches, not a non-sticky error that an earlier runtime call left behind (a sticky error of
// a faulted context still surfaces).
template <class F>
int launched(int n, F&& enqueue) {
  cudaGetLastError();
  enqueue();
  g_launches.fetch_add(n);
  CU(cudaGetLastError());
  return 0;
}

// Owners of CUDA resources.  Objects free their members on their own device: each destructor body below selects it,
// and member destructors run after the body.
struct CudaFree {
  void operator()(void* p) const { cudaFree(p); }
};
struct CudaFreeAsync {  // stream-ordered scratch
  cudaStream_t st;
  void operator()(void* p) const { cudaFreeAsync(p, st); }
};
struct StreamDestroy {
  void operator()(cudaStream_t s) const { cudaStreamDestroy(s); }
};
struct EventDestroy {
  void operator()(cudaEvent_t e) const { cudaEventDestroy(e); }
};
template <class T>
using DevBuf = std::unique_ptr<T, CudaFree>;
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;

// Frees what b holds, then allocates `bytes` into it; b stays empty on failure.
template <class T>
cudaError_t dev_alloc(DevBuf<T>& b, size_t bytes) {
  b.reset();
  void* p = nullptr;
  const cudaError_t e = cudaMalloc(&p, bytes);
  if (e == cudaSuccess) b.reset(static_cast<T*>(p));
  return e;
}
template <class T>
cudaError_t dev_upload(DevBuf<T>& b, const T* src, size_t n) {
  const cudaError_t e = dev_alloc(b, n * sizeof(T));
  return e == cudaSuccess ? cudaMemcpy(b.get(), src, n * sizeof(T), cudaMemcpyHostToDevice) : e;
}
cudaError_t make_stream(Stream& s) {
  cudaStream_t r = nullptr;
  const cudaError_t e = cudaStreamCreateWithFlags(&r, cudaStreamNonBlocking);
  s.reset(e == cudaSuccess ? r : nullptr);
  return e;
}
cudaError_t make_event(Event& ev, unsigned flags) {
  cudaEvent_t r = nullptr;
  const cudaError_t e = cudaEventCreateWithFlags(&r, flags);
  ev.reset(e == cudaSuccess ? r : nullptr);
  return e;
}

long long* g_dbg_ts = nullptr;  // timing experiments only (vadb200_debug_timestamps)
constexpr int kNumSmFallback = 148;
constexpr int kPlanCounters = 16;  // launches of one plan that may be in flight at once (any streams)
constexpr int kHostBufs = 3;
constexpr int kWinPairs = kFftN / 2;  // window pairs for any frame_len <= 512; entries past 400 stay 1

// One staging slot of the vad_host pipeline: the chunk's PCM, its results, and the events that order the slot's reuse.
struct HostBuf {
  DevBuf<int16_t> stage;
  DevBuf<uint8_t> labels;
  DevBuf<float> logits, rows;
  Event in, done, out;
};
// Grows one buffer of every staging slot to `count` elements; contents are not kept.
template <class T>
int grow(HostBuf (&slots)[kHostBufs], DevBuf<T> HostBuf::*buf, long long& cap, long long count) {
  if (count <= cap) return 0;
  cap = 0;  // a failure part way must not leave a capacity that some slot lacks
  for (HostBuf& s : slots) CU(dev_alloc(s.*buf, count * sizeof(T)));
  cap = count;
  return 0;
}

}  // namespace

struct vadb200_handle {
  ~vadb200_handle() { cudaSetDevice(device); }
  int device = 0;
  unsigned long long id = 0;
  unsigned version = 1;
  MfccConfig cfg;
  std::vector<double> fb;
  MelDctTables tab;   // identical for every handle (only the reference configuration is compiled in)
  FfnParams par;      // per-handle FFN weights: passed to kernels as a launch parameter
  FfnBias bias;       // the same biases for the tensor-core variant
  int plan_seg_frames = 0;  // 0 = automatic segment length (vadb200_set_plan_segment_frames)
  bool have_ffn = false;
  DevBuf<cf2> d_tw;  // tw1[256] then tw2[128]
  int num_sms = kNumSmFallback;
  long long host_chunk_samples = 32ll << 20;
  // vad_host pipeline resources (lazy): usable once all streams and events exist
  bool pipe_ready = false;
  Stream s_in, s_run, s_out;
  HostBuf hb[kHostBufs];
  long long stage_cap = 0, lab_cap = 0, lgt_cap = 0, rows_cap = 0;  // elements in each slot's buffer
  DevBuf<float> d_sink;
  DevBuf<unsigned char> d_tc_blob;      // canonical tf32 hi/lo weight blob (ffn_tc.cuh)
  DevBuf<unsigned char> d_tc16_blob;    // canonical fp16 hi/lo weight blob, statically scaled
  bool tc16_ok = false;                 // the fp16 scales are in range for this handle's weights
  int ffn_impl = 2;                     // 0: FP32 CUDA cores, 1: tcgen05 tf32 hi/lo, 2: tcgen05 fp16 hi/lo (default)
  // opt-in front end (vadb200_set_frontend); the decision threshold lives in par.thresh / bias.thresh
  float preemph = 0.0f;
  bool has_window = false;
  float window[kFrame] = {};
  DevBuf<cf2> d_win;                    // [kWinPairs] window pairs, all ones without a window (per handle: no globals)
};

struct vadb200_plan {
  ~vadb200_plan() { cudaSetDevice(device); }
  vadb200_handle* h = nullptr;
  int device = 0;                     // h->device, kept so destroy never reads a handle destroyed first
  int mode = 0;
  long long n_utt = 0;
  std::vector<long long> offsets, lengths, row_off, utt_seg;  // utt_seg: n_utt + 1
  std::vector<Segment> segs;
  DevBuf<Segment> d_segs;
  DevBuf<int> d_counter;      // kPlanCounters self-resetting (next segment, CTAs done) pairs
  std::atomic<unsigned> launch_seq{0};
  long long total_rows = 0;
  long long seg_frames = 0;
  // speech segments (MODE_VAD / MODE_DATASET): tiles of <= kSpeechTile rows of one utterance
  std::vector<SpeechTile> tiles;
  std::vector<int> utt_tile;          // n_utt + 1: first tile of each utterance
  long long max_speech_segs = 0;      // sum over utterances of ceil(R_u / 2)
  DevBuf<long long> d_row_off;        // n_utt + 1 row offsets
  DevBuf<long long> d_pcm_off;        // n_utt sample offsets
  DevBuf<SpeechTile> d_tiles;
  DevBuf<int> d_utt_tile;
};

struct vadb200_trainer {
  ~vadb200_trainer() { cudaSetDevice(device); }
  vadb200_handle* h = nullptr;
  int device = 0;              // h->device, kept so destroy never reads a handle destroyed first
  long long max_batch = 0;
  float lr = 1.0f, rho = 0.95f, eps = 1e-8f;
  DevBuf<float> d_state;       // params | acc_g | acc_u   (3 x kNParams)
  DevBuf<float> d_partial;     // [min(ceil(max_batch / 128), SMs)][kNParams + 1]
  DevBuf<float> d_loss;
  long long steps = 0;
};

struct vadb200_bank {
  ~vadb200_bank() { cudaSetDevice(device); }
  vadb200_handle* h = nullptr;
  int device = 0;              // h->device, kept so destroy never reads a handle destroyed first
  int n = 0;
  DevBuf<int16_t> d_hist;
  DevBuf<float> d_ring;
  DevBuf<int> d_fed;
  DevBuf<int16_t> d_prev;      // the raw sample before each stream's history (front end)
  // ragged bank (vadb200_stream_bank_create_ragged; max_feed == 0: the fixed bank, which has d_hist, d_fed, d_prev
  // instead): per stream a sample ring of ring_len int16 and the samples taken so far (vad_ragged.h)
  int max_feed = 0;
  int ring_len = 0;
  DevBuf<int16_t> d_pcm;
  DevBuf<long long> d_total;
  // speech segments (vadb200_stream_bank_set_speech); d_seg empty: off.  One allocation of
  // [W1 + W2 + 2][n] words: ring1, ring2, meta, last (vad_segments.cuh StreamSeg).
  SmoothParams sp{};
  DevBuf<uint32_t> d_seg;
  size_t seg_bytes = 0;
};

struct vadb200_resampler {
  ~vadb200_resampler() { cudaSetDevice(device); }
  int device = 0;
  int num_sms = kNumSmFallback;
  ResampleDesign d;
  DevBuf<float> d_taps;        // [up][Ks] float32 polyphase rows (vad_resample.cuh)
};

namespace {

bool frontend_on(const vadb200_handle* h) { return h->preemph != 0.0f || h->has_window; }
FrontEnd frontend_of(const vadb200_handle* h) { return FrontEnd{h->d_win.get(), h->preemph}; }

// The classifier a handle runs: 2 (tcgen05 fp16 hi/lo) when asked for and the weights fit its static scales, else
// 1 (tcgen05 tf32 hi/lo) when any tensor-core variant is asked for, else 0 (FP32 CUDA cores); and its weight blob.
struct Classifier {
  int tc;
  const unsigned char* blob;
};
Classifier classifier_of(const vadb200_handle* h) {
  if (h->ffn_impl == 2 && h->tc16_ok) return {2, h->d_tc16_blob.get()};
  if (h->ffn_impl >= 1) return {1, h->d_tc_blob.get()};
  return {0, nullptr};
}

template <int MODE, int TC>
void enqueue_fused(bool fe, int grid, cudaStream_t st, const FusedParams& fp,
                   const typename FfnArgOf<MODE, TC>::type& ffn, const FrontEnd& fea) {
  if (fe) fused_fe_kernel<MODE, TC><<<grid, kThreads, kFusedSmemBytes, st>>>(fp, ffn, fea);
  else fused_kernel<MODE, TC><<<grid, kThreads, kFusedSmemBytes, st>>>(fp, ffn);
}

int launch_fused(vadb200_plan* p, FusedParams fp, int n_segs, cudaStream_t st) {
  vadb200_handle* h = p->h;
  if (n_segs <= 0) return 0;
  // each launch takes its own self-resetting counter pair, so one plan can be in flight on several streams
  fp.counter = p->d_counter.get() + 2 * (p->launch_seq.fetch_add(1) % kPlanCounters);
#if defined(VADB_DEBUG_HOOKS)
  const char* gps = std::getenv("VADB200_CTAS_PER_SM");  // occupancy experiments only
  const int per_sm = gps ? std::max(1, std::atoi(gps)) : 2;
#else
  const int per_sm = 2;
#endif
  const int grid = std::min(n_segs, per_sm * h->num_sms);
  // the front-end variant runs only when the handle asks for a front end or (VAD) a decision threshold
  const bool fe = frontend_on(h) || (p->mode == VADB200_MODE_VAD && h->par.thresh > 0.0f);
  const FrontEnd fea = frontend_of(h);
  const Classifier c = classifier_of(h);
  if (p->mode == VADB200_MODE_VAD) fp.tc_blob = c.blob;
  return launched(1, [&] {
    if (p->mode == VADB200_MODE_MFCC) enqueue_fused<0, 0>(fe, grid, st, fp, FfnNone{0}, fea);
    else if (p->mode == VADB200_MODE_DATASET) enqueue_fused<1, 0>(fe, grid, st, fp, FfnNone{0}, fea);
    else if (c.tc == 2) enqueue_fused<2, 2>(fe, grid, st, fp, h->bias, fea);
    else if (c.tc == 1) enqueue_fused<2, 1>(fe, grid, st, fp, h->bias, fea);
    else enqueue_fused<2, 0>(fe, grid, st, fp, h->par, fea);
  });
}

FusedParams base_params(vadb200_plan* p) {
  FusedParams fp;
  std::memset(&fp, 0, sizeof(fp));
  fp.segs = p->d_segs.get();
  fp.counter = p->d_counter.get();  // launch_fused picks the launch's own pair
  fp.tw1 = p->h->d_tw.get();
  fp.tw2 = p->h->d_tw.get() + 256;
#if defined(VADB_DEBUG_HOOKS)
  const char* dbg = std::getenv("VADB200_DEBUG_SKIP");  // timing experiments only; results are garbage
  fp.debug_skip = dbg ? std::atoi(dbg) : 0;
  fp.dbg_ts = g_dbg_ts;
#else
  fp.debug_skip = 0;
  fp.dbg_ts = nullptr;
#endif
  return fp;
}

// The classifier crosses the C ABI as eight arrays W1, b1, ..., W4, b4; the kNParams parameter vector, which is also
// how FfnParams begins, holds them back to back from these offsets.
constexpr int kParamOff[9] = {kOffW1, kOffB1, kOffW2, kOffB2, kOffW3, kOffB3, kOffW4, kOffB4, kNParams};
static_assert(offsetof(FfnParams, thresh) == kNParams * sizeof(float), "FfnParams starts with the parameter vector");
void pack_params(const float* const (&src)[8], float* v) {
  for (int i = 0; i < 8; ++i) std::memcpy(v + kParamOff[i], src[i], (kParamOff[i + 1] - kParamOff[i]) * sizeof(float));
}
void unpack_params(const float* v, float* const (&dst)[8]) {
  for (int i = 0; i < 8; ++i) std::memcpy(dst[i], v + kParamOff[i], (kParamOff[i + 1] - kParamOff[i]) * sizeof(float));
}

}  // namespace

extern "C" {

const char* vadb200_last_error(void) { return g_err.c_str(); }
int vadb200_version(void) { return VADB200_VERSION; }
int64_t vadb200_launch_count(void) { return g_launches.load(); }
// Timing experiments only (not in the public header): device buffer of 64 x 16 clock64 stamps written by
// CTA 0 during its first block phases; pass NULL to switch off.
int vadb200_debug_timestamps(long long* d_buf) { g_dbg_ts = d_buf; return 0; }

void vadb200_default_config(vadb200_config* c) {
  if (!c) return;
  c->sample_rate = 16000; c->frame_size = 400; c->frame_step = 160; c->fft_n = 512;
  c->n_filters = 26; c->n_mfcc = 13; c->low_hz = 300.0; c->high_hz = 8000.0; c->lifter_l = 22;
  c->reserved = 0;
}

int64_t vadb200_frames_for_length(int64_t n) { return frames_for_length(n); }
int64_t vadb200_outputs_for_length(int64_t n) { return outputs_for_length(n); }

int vadb200_create(const vadb200_config* c, int device, vadb200_handle** out) {
  if (!out) return fail(VADB200_E_INVALID, "out is null");
  *out = nullptr;
  vadb200_config dc;
  if (!c) {
    vadb200_default_config(&dc);
    c = &dc;
  }
  MfccConfig cfg;
  cfg.sample_rate = c->sample_rate; cfg.frame_size = c->frame_size; cfg.frame_step = c->frame_step;
  cfg.fft_n = c->fft_n; cfg.n_filters = c->n_filters; cfg.n_mfcc = c->n_mfcc;
  cfg.low_hz = c->low_hz; cfg.high_hz = c->high_hz; cfg.lifter_l = c->lifter_l;
  if (!is_reference_config(cfg))
    return fail(VADB200_E_UNSUPPORTED,
                "only the reference configuration (16 kHz, 400/160, n_fft 512, 26 filters 300-8000 Hz, 13 "
                "cepstra, lifter 22; config.py:20-27) is compiled in");
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(VADB200_E_INVALID, "no such CUDA device");
  if (device >= 64) return fail(VADB200_E_INVALID, "device index >= 64");
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    return fail(VADB200_E_UNSUPPORTED, "kernels are built for sm_100a (B200) only");
  std::unique_ptr<vadb200_handle> h(new (std::nothrow) vadb200_handle());
  if (!h) return fail(VADB200_E_NOMEM, "host allocation failed");
  h->device = device;
  h->id = g_next_id.fetch_add(1);
  h->cfg = cfg;
  h->num_sms = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : kNumSmFallback;
  h->fb = mel_filterbank(cfg);
  std::fill(h->window, h->window + kFrame, 1.0f);  // rectangular
  std::memset(&h->par, 0, sizeof(FfnParams));
  std::memset(&h->bias, 0, sizeof(FfnBias));
  std::memset(&h->tab, 0, sizeof(MelDctTables));
  std::string why;
  if (!pack_mel_weights(h->fb.data(), h->tab.melw, &why)) return fail(VADB200_E_UNSUPPORTED, why);
  folded_dct(cfg, h->tab.dct);
  pack_mel_pairs(h->fb.data(), h->tab.melw2);
  pack_dct_pairs(h->tab.dct, h->tab.dctp);
  cf2 tw[384];
  fft_twiddles(tw, tw + 256);
  CU(dev_upload(h->d_tw, tw, 384));
  CU(dev_alloc(h->d_sink, 256));
  CU(dev_alloc(h->d_tc_blob, kTcBlobBytes));
  CU(dev_alloc(h->d_tc16_blob, kTc16BlobBytes));
  const std::vector<cf2> ones(kWinPairs, cf2{1.0f, 1.0f});
  CU(dev_upload(h->d_win, ones.data(), kWinPairs));
  // function attributes and the (config-invariant) constant tables now, so that no launch ever
  // synchronises: every device-pointer entry point can be captured into a CUDA graph
  CU(cudaFuncSetAttribute(fused_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmemBytes));
  CU(cudaFuncSetAttribute(fused_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmemBytes));
  CU(cudaFuncSetAttribute(fused_kernel<2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmemBytes));
  CU(cudaFuncSetAttribute(fused_kernel<2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmemBytes));
  CU(cudaFuncSetAttribute(fused_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmemBytes));
  CU(cudaFuncSetAttribute(fused_fe_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmemBytes));
  CU(cudaFuncSetAttribute(fused_fe_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmemBytes));
  CU(cudaFuncSetAttribute(fused_fe_kernel<2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmemBytes));
  CU(cudaFuncSetAttribute(fused_fe_kernel<2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmemBytes));
  CU(cudaFuncSetAttribute(fused_fe_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedSmemBytes));
  CU(cudaFuncSetAttribute(ffn_tc_rows_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFfnTcSmemBytes));
  CU(cudaFuncSetAttribute(ffn_tc_rows_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFfnTcSmemBytes));
  CU(cudaFuncSetAttribute(frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFramesSmemBytes));
  CU(cudaFuncSetAttribute(stream_feed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStreamSmemBytes));
  CU(cudaFuncSetAttribute(stream_feed_speech_kernel<StreamSeg>, cudaFuncAttributeMaxDynamicSharedMemorySize, kStreamSmemBytes));
  CU(cudaFuncSetAttribute(stream_ragged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStreamSmemBytes));
  CU(cudaFuncSetAttribute(stream_ragged_speech_kernel<StreamSeg>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          kStreamSmemBytes));
  // Mel weights and the folded DCT matrix are the same for every handle (the kernels are compiled for the
  // reference configuration only), so the __constant__ copy is written once per device and never changes:
  // no handle can observe another handle's state through it.  FFN weights never go through device globals.
  {
    std::lock_guard<std::mutex> lk(g_tab_mu);
    if (!g_tab_loaded[device]) {
      CU(cudaMemcpyToSymbol(c_tab, &h->tab, sizeof(MelDctTables), 0, cudaMemcpyHostToDevice));
      CU(cudaDeviceSynchronize());
      g_tab_loaded[device] = true;
    }
  }
  *out = h.release();
  return 0;
}

int vadb200_destroy(vadb200_handle* h) {
  delete h;
  return 0;
}

int vadb200_get_filterbank(vadb200_handle* h, double* out) {
  if (!h || !out) return fail(VADB200_E_INVALID, "null argument");
  std::memcpy(out, h->fb.data(), h->fb.size() * sizeof(double));
  return 0;
}

int vadb200_set_ffn_weights(vadb200_handle* h, const float* W1, const float* b1, const float* W2, const float* b2,
                            const float* W3, const float* b3, const float* W4, const float* b4) {
  const float* src[8] = {W1, b1, W2, b2, W3, b3, W4, b4};
  if (!h || std::count(src, src + 8, nullptr)) return fail(VADB200_E_INVALID, "null argument");
  std::vector<float> v(kNParams);
  pack_params(src, v.data());
  std::memcpy(&h->par, v.data(), kNParams * sizeof(float));
  std::memcpy(h->bias.b1, b1, sizeof(h->bias.b1)); std::memcpy(h->bias.b2, b2, sizeof(h->bias.b2));
  std::memcpy(h->bias.b3, b3, sizeof(h->bias.b3)); std::memcpy(h->bias.b4, b4, sizeof(h->bias.b4));
  h->have_ffn = true;
  h->version = (h->version + 1) & 0xFFFFF;
  // tensor-core operand blob; drained + blocking so kernels on any stream see a consistent copy
  std::vector<unsigned char> blob(kTcBlobBytes);
  tc_pack_weights(h->par, blob.data());
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(h->d_tc_blob.get(), blob.data(), kTcBlobBytes, cudaMemcpyHostToDevice));
  std::vector<unsigned char> blob16(kTc16BlobBytes);
  h->tc16_ok = tc16_pack_weights(h->par, blob16.data(), h->bias);
  if (h->tc16_ok) CU(cudaMemcpy(h->d_tc16_blob.get(), blob16.data(), kTc16BlobBytes, cudaMemcpyHostToDevice));
  return 0;
}

int vadb200_set_ffn_impl(vadb200_handle* h, int impl) {
  if (!h || impl < 0 || impl > 2)
    return fail(VADB200_E_INVALID, "impl must be 0 (fp32), 1 (tcgen05 tf32 hi/lo) or 2 (tcgen05 fp16 hi/lo)");
  h->ffn_impl = impl;
  return 0;
}
int vadb200_get_ffn_impl(vadb200_handle* h) { return h ? h->ffn_impl : -1; }

int vadb200_set_frontend(vadb200_handle* h, float preemph, const float* h_window) {
  if (!h) return fail(VADB200_E_INVALID, "handle is null");
  if (!(preemph >= 0.0f && preemph <= 1.0f)) return fail(VADB200_E_INVALID, "pre-emphasis must be in [0, 1]");
  if (h_window)
    for (int i = 0; i < kFrame; ++i)
      if (!std::isfinite(h_window[i])) return fail(VADB200_E_INVALID, "window weights must be finite");
  std::vector<cf2> pairs(kWinPairs, cf2{1.0f, 1.0f});
  if (h_window)
    for (int m = 0; m < kFrame / 2; ++m) pairs[m] = cf2{h_window[2 * m], h_window[2 * m + 1]};
  // drained + blocking, like the FFN weights: kernels on any stream see a consistent table
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(h->d_win.get(), pairs.data(), kWinPairs * sizeof(cf2), cudaMemcpyHostToDevice));
  h->preemph = preemph;
  h->has_window = h_window != nullptr;
  if (h_window) std::memcpy(h->window, h_window, sizeof(h->window));
  else std::fill(h->window, h->window + kFrame, 1.0f);
  return 0;
}

int vadb200_get_frontend(vadb200_handle* h, float* preemph, float* h_window, int* has_window) {
  if (!h) return fail(VADB200_E_INVALID, "handle is null");
  if (preemph) *preemph = h->preemph;
  if (has_window) *has_window = h->has_window ? 1 : 0;
  if (h_window) std::memcpy(h_window, h->window, sizeof(h->window));
  return 0;
}

int vadb200_set_decision_threshold(vadb200_handle* h, float p_voiced) {
  if (!h) return fail(VADB200_E_INVALID, "handle is null");
  if (!(p_voiced < 1.0f)) return fail(VADB200_E_INVALID, "threshold must be < 1 (<= 0: argmax)");
  const float th = p_voiced > 0.0f ? p_voiced : 0.0f;
  h->par.thresh = th;
  h->bias.thresh = th;
  return 0;
}

float vadb200_get_decision_threshold(vadb200_handle* h) { return h ? h->par.thresh : NAN; }

int vadb200_set_host_chunk_samples(vadb200_handle* h, int64_t samples) {
  if (!h || samples < 4096) return fail(VADB200_E_INVALID, "chunk must be >= 4096 samples");
  h->host_chunk_samples = samples & ~7ll;
  return 0;
}

// ---- plans ---------------------------------------------------------------------------------------------
int vadb200_plan_create(vadb200_handle* h, const int64_t* offs, const int64_t* lens, int64_t n_utt, int mode,
                        vadb200_plan** out) {
  if (!h || !out || n_utt < 0 || (n_utt > 0 && (!offs || !lens))) return fail(VADB200_E_INVALID, "null / negative argument");
  if (mode < 0 || mode > 2) return fail(VADB200_E_INVALID, "unknown mode");
  *out = nullptr;
  std::unique_ptr<vadb200_plan> p(new (std::nothrow) vadb200_plan());
  if (!p) return fail(VADB200_E_NOMEM, "host allocation failed");
  p->h = h; p->device = h->device; p->mode = mode; p->n_utt = n_utt;
  p->offsets.assign(offs, offs + n_utt);
  p->lengths.assign(lens, lens + n_utt);
  p->row_off.resize(n_utt + 1);
  p->utt_seg.resize(n_utt + 1);
  long long rows = 0, prev_end = 0;
  for (long long u = 0; u < n_utt; ++u) {
    if (offs[u] < 0 || (offs[u] & 7) || lens[u] < 0 || offs[u] < prev_end)
      return fail(VADB200_E_INVALID, "utterance offsets must be ascending, non-overlapping multiples of 8 samples");
    prev_end = offs[u] + lens[u];
    p->row_off[u] = rows;
    rows += (mode == VADB200_MODE_MFCC) ? frames_for_length(lens[u]) : outputs_for_length(lens[u]);
  }
  p->row_off[n_utt] = rows;
  p->total_rows = rows;
  // Segment length: long runs amortise the 4-frame halo; short ones keep all CTAs busy on small
  // batches.  n_frames of a full segment is a multiple of 32 (whole steps).
  const int halo = (mode == VADB200_MODE_MFCC) ? 0 : 4;
  long long seg_frames = h->plan_seg_frames;
  if (seg_frames <= 0) {
    // >= 16 segments per persistent CTA when the batch allows (dynamic scheduling then balances to a few
    // per cent), whole 128-frame tensor-core tiles, at most 2048 frames
    const long long want = rows / (16ll * 2 * h->num_sms) + halo;
    seg_frames = want <= 64 ? 64 : std::min<long long>(2048, ((want + 127) / 128) * 128);
  }
  p->seg_frames = seg_frames;
  const long long seg_rows = seg_frames - halo;
  for (long long u = 0; u < n_utt; ++u) {
    p->utt_seg[u] = static_cast<long long>(p->segs.size());
    const long long r = p->row_off[u + 1] - p->row_off[u];
    for (long long o = 0; o < r; o += seg_rows) {
      Segment s;
      s.pcm_start = offs[u] + kHop * o;
      s.out_start = p->row_off[u] + o;
      s.n_frames = static_cast<int>(std::min(seg_rows, r - o) + halo);
      s.cont = o > 0 ? 1 : 0;
      p->segs.push_back(s);
    }
  }
  p->utt_seg[n_utt] = static_cast<long long>(p->segs.size());
  if (p->segs.size() > 0x7fffffffull) return fail(VADB200_E_INVALID, "too many segments");
  if (mode != VADB200_MODE_MFCC) {
    p->utt_tile.resize(n_utt + 1);
    for (long long u = 0; u < n_utt; ++u) {
      p->utt_tile[u] = static_cast<int>(p->tiles.size());
      const long long r = p->row_off[u + 1] - p->row_off[u];
      p->max_speech_segs += (r + 1) / 2;
      for (long long o = 0; o < r; o += kSpeechTile)
        p->tiles.push_back(SpeechTile{p->row_off[u] + o, static_cast<int>(std::min<long long>(kSpeechTile, r - o)),
                                      static_cast<int>(u)});
    }
    p->utt_tile[n_utt] = static_cast<int>(p->tiles.size());
  }
  CU(cudaSetDevice(h->device));
  CU(dev_alloc(p->d_counter, 2 * kPlanCounters * sizeof(int)));
  CU(cudaMemset(p->d_counter.get(), 0, 2 * kPlanCounters * sizeof(int)));
  if (!p->segs.empty()) CU(dev_upload(p->d_segs, p->segs.data(), p->segs.size()));
  if (mode != VADB200_MODE_MFCC) {
    CU(dev_upload(p->d_row_off, p->row_off.data(), n_utt + 1));
    CU(dev_upload(p->d_utt_tile, p->utt_tile.data(), n_utt + 1));
    if (n_utt > 0) CU(dev_upload(p->d_pcm_off, p->offsets.data(), n_utt));
    if (!p->tiles.empty()) CU(dev_upload(p->d_tiles, p->tiles.data(), p->tiles.size()));
  }
  *out = p.release();
  return 0;
}

int vadb200_plan_destroy(vadb200_plan* p) {
  delete p;
  return 0;
}

int64_t vadb200_plan_total_rows(const vadb200_plan* p) { return p ? p->total_rows : -1; }
int64_t vadb200_plan_segment_frames(const vadb200_plan* p) { return p ? p->seg_frames : -1; }
int64_t vadb200_plan_segment_count(const vadb200_plan* p) { return p ? static_cast<int64_t>(p->segs.size()) : -1; }

int vadb200_set_plan_segment_frames(vadb200_handle* h, int frames) {
  if (!h || frames < 0 || frames > 2048 || (frames != 0 && (frames < 64 || frames % 32)))
    return fail(VADB200_E_INVALID, "segment length must be 0 (automatic) or a multiple of 32 in [64, 2048]");
  h->plan_seg_frames = frames;
  return 0;
}

int vadb200_plan_row_offsets(const vadb200_plan* p, int64_t* out) {
  if (!p || !out) return fail(VADB200_E_INVALID, "null argument");
  for (long long u = 0; u <= p->n_utt; ++u) out[u] = p->row_off[u];
  return 0;
}

static int check_pcm(const vadb200_plan* p, const void* pcm, int64_t pcm_len) {
  if (!p) return fail(VADB200_E_INVALID, "plan is null");
  if (p->total_rows > 0 && !pcm) return fail(VADB200_E_INVALID, "pcm is null");
  if (reinterpret_cast<uintptr_t>(pcm) & 15) return fail(VADB200_E_INVALID, "pcm must be 16-byte aligned");
  if (p->n_utt > 0 && pcm_len < p->offsets[p->n_utt - 1] + p->lengths[p->n_utt - 1])
    return fail(VADB200_E_INVALID, "pcm_len is smaller than the last utterance's end");
  return 0;
}

int vadb200_mfcc_packed(vadb200_plan* p, const int16_t* d_pcm, int64_t pcm_len, float* d_out, void* stream) {
  int rc = check_pcm(p, d_pcm, pcm_len);
  if (rc) return rc;
  if (p->mode == VADB200_MODE_VAD) return fail(VADB200_E_INVALID, "plan was created for MODE_VAD");
  if (p->total_rows > 0 && !d_out) return fail(VADB200_E_INVALID, "d_out is null");
  CU(cudaSetDevice(p->h->device));
  FusedParams fp = base_params(p);
  fp.pcm = d_pcm; fp.pcm_len = pcm_len; fp.rows = d_out;
  fp.seg_begin = 0; fp.seg_end = static_cast<int>(p->segs.size());
  return launch_fused(p, fp, fp.seg_end, static_cast<cudaStream_t>(stream));
}

int vadb200_vad_packed(vadb200_plan* p, const int16_t* d_pcm, int64_t pcm_len, uint8_t* d_labels, float* d_logits,
                       float* d_feats, int feat_mode, void* stream) {
  int rc = check_pcm(p, d_pcm, pcm_len);
  if (rc) return rc;
  if (p->mode != VADB200_MODE_VAD) return fail(VADB200_E_INVALID, "plan was not created for MODE_VAD");
  if (!p->h->have_ffn) return fail(VADB200_E_STATE, "FFN weights not set (vadb200_set_ffn_weights)");
  if (p->total_rows > 0 && !d_labels) return fail(VADB200_E_INVALID, "d_labels is null");
  if (feat_mode != VADB200_FEAT_ANALYSER && feat_mode != VADB200_FEAT_DATASET) return fail(VADB200_E_INVALID, "unknown feat_mode");
  CU(cudaSetDevice(p->h->device));
  FusedParams fp = base_params(p);
  fp.pcm = d_pcm; fp.pcm_len = pcm_len; fp.labels = d_labels; fp.logits = d_logits; fp.feats = d_feats;
  fp.feat_mode = feat_mode;
  fp.seg_begin = 0; fp.seg_end = static_cast<int>(p->segs.size());
  return launch_fused(p, fp, fp.seg_end, static_cast<cudaStream_t>(stream));
}

// ---- host-buffer pipeline ---------------------------------------------------------------------------------
static int ensure_host_pipeline(vadb200_handle* h, long long stage_samples, long long rows, bool want_labels,
                                bool want_logits, long long row_floats) {
  if (!h->pipe_ready) {
    for (Stream* s : {&h->s_in, &h->s_run, &h->s_out}) CU(make_stream(*s));
    for (HostBuf& s : h->hb)
      for (Event* ev : {&s.in, &s.done, &s.out}) CU(make_event(*ev, cudaEventDisableTiming));
    h->pipe_ready = true;
  }
  int rc = grow(h->hb, &HostBuf::stage, h->stage_cap, stage_samples);
  if (!rc && want_labels) rc = grow(h->hb, &HostBuf::labels, h->lab_cap, rows);
  if (!rc && want_logits) rc = grow(h->hb, &HostBuf::logits, h->lgt_cap, rows * 3);
  if (!rc) rc = grow(h->hb, &HostBuf::rows, h->rows_cap, row_floats);
  return rc;
}

// Chunked H2D -> fused kernel -> D2H over three staging buffers and three streams.  VAD plans return
// labels (+ logits); MFCC / dataset plans return float rows of `width` columns.
static int run_host_pipeline(vadb200_plan* p, const int16_t* h_pcm, int64_t pcm_len, uint8_t* h_labels, float* h_logits,
                             float* h_rows, int feat_mode) {
  vadb200_handle* h = p->h;
  if (p->total_rows == 0) return 0;
  if (p->n_utt > 0 && pcm_len < p->offsets[p->n_utt - 1] + p->lengths[p->n_utt - 1])
    return fail(VADB200_E_INVALID, "pcm_len is smaller than the last utterance's end");
  CU(cudaSetDevice(h->device));
  const long long width = p->mode == VADB200_MODE_VAD ? 0 : (p->mode == VADB200_MODE_MFCC ? kNCep : kNFeat);
  // chunks = runs of whole utterances whose PCM span fits host_chunk_samples
  struct Chunk { long long u0, u1, s0, s1; };
  std::vector<Chunk> chunks;
  long long max_span = 0, max_rows = 0;
  for (long long u = 0; u < p->n_utt;) {
    Chunk c{u, u, p->offsets[u], 0};
    while (c.u1 < p->n_utt && (c.u1 == c.u0 || p->offsets[c.u1] + p->lengths[c.u1] - c.s0 <= h->host_chunk_samples)) ++c.u1;
    c.s1 = p->offsets[c.u1 - 1] + p->lengths[c.u1 - 1];
    max_span = std::max(max_span, c.s1 - c.s0);
    max_rows = std::max(max_rows, p->row_off[c.u1] - p->row_off[c.u0]);
    chunks.push_back(c);
    u = c.u1;
  }
  max_rows = std::max<long long>(max_rows, 1);
  int rc = ensure_host_pipeline(h, ((max_span + 7) & ~7ll) + 8, max_rows, h_labels != nullptr, h_logits != nullptr,
                                width * max_rows);
  if (rc) return rc;
  cudaStream_t s_in = h->s_in.get(), s_run = h->s_run.get(), s_out = h->s_out.get();
  for (size_t i = 0; i < chunks.size(); ++i) {
    const Chunk& c = chunks[i];
    const HostBuf& slot = h->hb[i % kHostBufs];
    const long long span = c.s1 - c.s0;
    const long long r0 = p->row_off[c.u0], nrows = p->row_off[c.u1] - r0;
    if (i >= kHostBufs) CU(cudaStreamWaitEvent(s_in, slot.done.get(), 0));  // stage buffer free again
    CU(cudaMemcpyAsync(slot.stage.get(), h_pcm + c.s0, span * sizeof(int16_t), cudaMemcpyHostToDevice, s_in));
    CU(cudaEventRecord(slot.in.get(), s_in));
    CU(cudaStreamWaitEvent(s_run, slot.in.get(), 0));
    if (i >= kHostBufs) CU(cudaStreamWaitEvent(s_run, slot.out.get(), 0));  // result buffers drained
    FusedParams fp = base_params(p);
    fp.pcm = slot.stage.get() - c.s0;  // segment sample indices stay absolute
    fp.pcm_len = c.s1;
    fp.labels = h_labels ? slot.labels.get() : nullptr;
    fp.logits = h_logits ? slot.logits.get() : nullptr;
    fp.rows = width ? slot.rows.get() : nullptr;
    fp.row_base = r0;
    fp.feat_mode = feat_mode;
    fp.seg_begin = static_cast<int>(p->utt_seg[c.u0]);
    fp.seg_end = static_cast<int>(p->utt_seg[c.u1]);
    rc = launch_fused(p, fp, fp.seg_end - fp.seg_begin, s_run);
    if (rc) return rc;
    CU(cudaEventRecord(slot.done.get(), s_run));
    CU(cudaStreamWaitEvent(s_out, slot.done.get(), 0));
    if (nrows > 0) {
      if (h_labels) CU(cudaMemcpyAsync(h_labels + r0, slot.labels.get(), nrows, cudaMemcpyDeviceToHost, s_out));
      if (h_logits)
        CU(cudaMemcpyAsync(h_logits + r0 * 3, slot.logits.get(), nrows * 3 * sizeof(float), cudaMemcpyDeviceToHost,
                           s_out));
      if (width)
        CU(cudaMemcpyAsync(h_rows + r0 * width, slot.rows.get(), nrows * width * sizeof(float), cudaMemcpyDeviceToHost,
                           s_out));
    }
    CU(cudaEventRecord(slot.out.get(), s_out));
  }
  CU(cudaStreamSynchronize(s_out));
  CU(cudaStreamSynchronize(s_run));
  return 0;
}

int vadb200_vad_host(vadb200_plan* p, const int16_t* h_pcm, int64_t pcm_len, uint8_t* h_labels, float* h_logits,
                     int feat_mode) {
  if (!p) return fail(VADB200_E_INVALID, "plan is null");
  if (p->mode != VADB200_MODE_VAD) return fail(VADB200_E_INVALID, "plan was not created for MODE_VAD");
  if (!p->h->have_ffn) return fail(VADB200_E_STATE, "FFN weights not set (vadb200_set_ffn_weights)");
  if (feat_mode != VADB200_FEAT_ANALYSER && feat_mode != VADB200_FEAT_DATASET) return fail(VADB200_E_INVALID, "unknown feat_mode");
  if (p->total_rows == 0) return 0;
  if (!h_pcm || !h_labels) return fail(VADB200_E_INVALID, "null argument");
  return run_host_pipeline(p, h_pcm, pcm_len, h_labels, h_logits, nullptr, feat_mode);
}

int vadb200_mfcc_host(vadb200_plan* p, const int16_t* h_pcm, int64_t pcm_len, float* h_out) {
  if (!p) return fail(VADB200_E_INVALID, "plan is null");
  if (p->mode == VADB200_MODE_VAD) return fail(VADB200_E_INVALID, "plan was created for MODE_VAD");
  if (p->total_rows == 0) return 0;
  if (!h_pcm || !h_out) return fail(VADB200_E_INVALID, "null argument");
  return run_host_pipeline(p, h_pcm, pcm_len, nullptr, nullptr, h_out, 0);
}

// ---- feature sink / ingest -------------------------------------------------------------------------------
int vadb200_scale_rows(vadb200_handle* h, float* d_rows, int64_t n_rows, double* h_stats, void* stream) {
  if (!h || n_rows < 0) return fail(VADB200_E_INVALID, "bad argument");
  if (n_rows == 0) return 0;
  if (!d_rows) return fail(VADB200_E_INVALID, "d_rows is null");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double* scratch = nullptr;
  CU(cudaMallocAsync(&scratch, 6 * sizeof(double), st));  // stream-ordered scratch: no per-handle state
  const std::unique_ptr<double, CudaFreeAsync> acc(scratch, CudaFreeAsync{st});
  CU(cudaMemsetAsync(acc.get(), 0, 6 * sizeof(double), st));
  const long long total = n_rows * kNFeat;
  const int grid = static_cast<int>(std::min<long long>((total + 255) / 256, 8ll * h->num_sms));
  const int rc = launched(3, [&] {
    for (int pass = 0; pass < 3; ++pass) scale_rows_kernel<<<grid, 256, 0, st>>>(d_rows, n_rows, pass, acc.get());
  });
  if (rc) return rc;
  if (h_stats) {
    double raw[6];
    CU(cudaMemcpyAsync(raw, acc.get(), sizeof(raw), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const double cnt = static_cast<double>(n_rows) * kNCep;
    for (int g = 0; g < 3; ++g) {
      h_stats[g] = raw[g] / cnt;
      h_stats[3 + g] = std::sqrt(raw[3 + g] / cnt);
    }
  }
  return 0;
}

int vadb200_ingest_pcm(vadb200_handle* h, const void* d_raw, int big_endian, const int64_t* d_src_start,
                       const int64_t* d_dst_start, const int64_t* d_len, int n_seg, int64_t max_len, int16_t* d_dst,
                       void* stream) {
  if (!h || n_seg < 0 || max_len < 0) return fail(VADB200_E_INVALID, "bad argument");
  if (n_seg == 0 || max_len == 0) return 0;
  if (!d_raw || !d_src_start || !d_dst_start || !d_len || !d_dst) return fail(VADB200_E_INVALID, "null argument");
  if (reinterpret_cast<uintptr_t>(d_raw) & 1) return fail(VADB200_E_INVALID, "raw sample stream must be 2-byte aligned");
  if (n_seg > 65535) return fail(VADB200_E_INVALID, "at most 65535 segments per call");
  CU(cudaSetDevice(h->device));
  const unsigned gx = static_cast<unsigned>(std::min<long long>((max_len + 255) / 256, 4ll * h->num_sms));
  static_assert(sizeof(long long) == sizeof(int64_t), "int64_t layout");
  return launched(1, [&] {
    ingest_kernel<<<dim3(gx, static_cast<unsigned>(n_seg)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const uint8_t*>(d_raw), big_endian, reinterpret_cast<const long long*>(d_src_start),
        reinterpret_cast<const long long*>(d_dst_start), reinterpret_cast<const long long*>(d_len), d_dst);
  });
}

// ---- per-frame API ---------------------------------------------------------------------------------------
static int frames_common(vadb200_handle* h, const float* d_frames, int64_t n, int frame_len, int what, float* d_out,
                         void* stream) {
  if (!h) return fail(VADB200_E_INVALID, "handle is null");
  if (n < 0 || frame_len < 1 || frame_len > kFftN) return fail(VADB200_E_INVALID, "need 1 <= frame_len <= 512, n >= 0");
  if (h->has_window && frame_len != kFrame) return fail(VADB200_E_INVALID, "a window needs frame_len == 400");
  if (n == 0) return 0;
  if (!d_frames || !d_out) return fail(VADB200_E_INVALID, "null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned grid = static_cast<unsigned>((n + kStepFrames - 1) / kStepFrames);
  const FrontEnd fe = frontend_on(h) ? frontend_of(h) : FrontEnd{nullptr, 0.0f};
  const cf2* tw = h->d_tw.get();
  return launched(1, [&] {
    frames_kernel<<<grid, kThreads, kFramesSmemBytes, st>>>(d_frames, n, frame_len, what, d_out, tw, tw + 256, fe);
  });
}

int vadb200_spec_frames(vadb200_handle* h, const float* d_frames, int64_t n, int frame_len, float* d_spec, void* stream) {
  return frames_common(h, d_frames, n, frame_len, 0, d_spec, stream);
}
int vadb200_mfcc_frames(vadb200_handle* h, const float* d_frames, int64_t n, int frame_len, float* d_mfcc, void* stream) {
  return frames_common(h, d_frames, n, frame_len, 1, d_mfcc, stream);
}

int vadb200_mfcc_from_spec(vadb200_handle* h, const float* d_spec, int64_t n, float* d_mfcc, void* stream) {
  if (!h) return fail(VADB200_E_INVALID, "handle is null");
  if (n < 0) return fail(VADB200_E_INVALID, "n < 0");
  if (n == 0) return 0;
  if (!d_spec || !d_mfcc) return fail(VADB200_E_INVALID, "null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned grid = static_cast<unsigned>((n + kStepFrames - 1) / kStepFrames);
  return launched(1, [&] { spec_to_mfcc_kernel<<<grid, kThreads, 0, st>>>(d_spec, n, d_mfcc); });
}

int vadb200_vad_windows(vadb200_handle* h, const float* d_win, int64_t n, int feat_mode, uint8_t* d_labels,
                        float* d_logits, float* d_feats, void* stream) {
  if (!h) return fail(VADB200_E_INVALID, "handle is null");
  if (!h->have_ffn) return fail(VADB200_E_STATE, "FFN weights not set (vadb200_set_ffn_weights)");
  if (n < 0) return fail(VADB200_E_INVALID, "n < 0");
  if (n == 0) return 0;
  if (!d_win) return fail(VADB200_E_INVALID, "null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return launched(1, [&] {
    windows_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, st>>>(d_win, n, feat_mode, d_labels, d_logits,
                                                                         d_feats, h->par);
  });
}

int vadb200_ffn_predict(vadb200_handle* h, const float* d_x, int64_t n, uint8_t* d_labels, float* d_logits, void* stream) {
  if (!h) return fail(VADB200_E_INVALID, "handle is null");
  if (!h->have_ffn) return fail(VADB200_E_STATE, "FFN weights not set (vadb200_set_ffn_weights)");
  if (n < 0) return fail(VADB200_E_INVALID, "n < 0");
  if (n == 0) return 0;
  if (!d_x) return fail(VADB200_E_INVALID, "null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned grid = static_cast<unsigned>((n + 127) / 128);
  const Classifier c = classifier_of(h);
  return launched(1, [&] {
    // a fp16 tile holding a row past the feature bounds runs on the tf32 blob
    if (c.tc == 2)
      ffn_tc_rows_kernel<2><<<grid, 128, kFfnTcSmemBytes, st>>>(d_x, n, c.blob, h->d_tc_blob.get(), d_labels, d_logits,
                                                               h->bias);
    else if (c.tc == 1)
      ffn_tc_rows_kernel<1><<<grid, 128, kFfnTcSmemBytes, st>>>(d_x, n, nullptr, c.blob, d_labels, d_logits, h->bias);
    else
      ffn_rows_kernel<<<grid, 128, 0, st>>>(d_x, n, d_labels, d_logits, h->par);
  });
}

int vadb200_get_deltas(vadb200_handle* h, const float* d_a, const float* d_b, int64_t n, float* d_out, void* stream) {
  if (!h || n < 0) return fail(VADB200_E_INVALID, "bad argument");
  if (n == 0) return 0;
  if (!d_a || !d_b || !d_out) return fail(VADB200_E_INVALID, "null argument");
  CU(cudaSetDevice(h->device));
  return launched(1, [&] {
    elementwise_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        0, d_a, d_b, n, 1, 0, d_out);
  });
}

int vadb200_lifter(vadb200_handle* h, const float* d_in, int64_t n_rows, int ncoef, int L, float* d_out, void* stream) {
  if (!h || n_rows < 0 || ncoef < 1) return fail(VADB200_E_INVALID, "bad argument");
  if (n_rows == 0) return 0;
  if (!d_in || !d_out) return fail(VADB200_E_INVALID, "null argument");
  CU(cudaSetDevice(h->device));
  const long long n = n_rows * ncoef;
  return launched(1, [&] {
    elementwise_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        1, d_in, nullptr, n, ncoef, L, d_out);
  });
}

// ---- streaming -------------------------------------------------------------------------------------------
int vadb200_stream_bank_create(vadb200_handle* h, int n_streams, vadb200_bank** out) {
  if (!h || !out || n_streams < 1) return fail(VADB200_E_INVALID, "bad argument");
  *out = nullptr;
  CU(cudaSetDevice(h->device));
  std::unique_ptr<vadb200_bank> b(new (std::nothrow) vadb200_bank());
  if (!b) return fail(VADB200_E_NOMEM, "host allocation failed");
  b->h = h; b->device = h->device; b->n = n_streams;
  CU(dev_alloc(b->d_hist, static_cast<size_t>(n_streams) * 320 * sizeof(int16_t)));
  CU(dev_alloc(b->d_ring, static_cast<size_t>(n_streams) * 5 * kNCep * sizeof(float)));
  CU(dev_alloc(b->d_fed, static_cast<size_t>(n_streams) * sizeof(int)));
  CU(dev_alloc(b->d_prev, static_cast<size_t>(n_streams) * sizeof(int16_t)));
  const int rc = vadb200_stream_bank_reset(b.get(), nullptr);
  if (rc) return rc;
  CU(cudaDeviceSynchronize());  // state is zero before any stream can feed
  *out = b.release();
  return 0;
}

int vadb200_stream_bank_create_ragged(vadb200_handle* h, int n_streams, int max_feed_samples, vadb200_bank** out) {
  if (out) *out = nullptr;
  if (!h || !out || n_streams < 1 || max_feed_samples < 1 || max_feed_samples > kRaggedMaxFeed)
    return fail(VADB200_E_INVALID, "bad argument (max_feed_samples must lie in [1, 16000])");
  CU(cudaSetDevice(h->device));
  std::unique_ptr<vadb200_bank> b(new (std::nothrow) vadb200_bank());
  if (!b) return fail(VADB200_E_NOMEM, "host allocation failed");
  b->h = h; b->device = h->device; b->n = n_streams;
  b->max_feed = max_feed_samples;
  b->ring_len = ragged_ring_samples(max_feed_samples);
  CU(dev_alloc(b->d_pcm, static_cast<size_t>(n_streams) * b->ring_len * sizeof(int16_t)));
  CU(dev_alloc(b->d_total, static_cast<size_t>(n_streams) * sizeof(long long)));
  CU(dev_alloc(b->d_ring, static_cast<size_t>(n_streams) * 5 * kNCep * sizeof(float)));
  const int rc = vadb200_stream_bank_reset(b.get(), nullptr);
  if (rc) return rc;
  CU(cudaDeviceSynchronize());  // state is zero before any stream can feed
  *out = b.release();
  return 0;
}

int vadb200_stream_bank_max_rows_per_feed(const vadb200_bank* b) {
  return b && b->max_feed ? ragged_max_rows(b->max_feed) : -1;
}

int vadb200_stream_bank_destroy(vadb200_bank* b) {
  delete b;
  return 0;
}

namespace {

StreamSeg bank_seg(const vadb200_bank* b, uint8_t* d_rows, int64_t* d_bounds) {
  StreamSeg g{};
  if (!b->d_seg) return g;
  const SmoothParams& sp = b->sp;
  g.n = b->n;
  g.G = sp.G; g.S = sp.S; g.P = sp.P; g.H = sp.H;
  g.d1 = sp.G > 1 ? sp.G - 1 : 0;
  g.d2 = sp.S > 1 ? sp.S - 1 : 0;
  const long long w1 = g.d1 ? seg_ring_words(g.d1) : 0, w2 = g.d2 ? seg_ring_words(g.d2) : 0;
  g.ring1 = b->d_seg.get();
  g.ring2 = b->d_seg.get() + w1 * b->n;
  g.meta = b->d_seg.get() + (w1 + w2) * b->n;
  g.last = reinterpret_cast<int*>(g.meta + b->n);
  g.rows = d_rows;
  g.bounds = d_bounds;
  return g;
}

int launch_stream_feed(vadb200_bank* b, const int16_t* d_chunks, uint8_t* d_labels, float* d_logits, uint8_t* d_rows,
                       int64_t* d_bounds, void* stream) {
  if (!b || !d_chunks || !d_labels) return fail(VADB200_E_INVALID, "null argument");
  vadb200_handle* h = b->h;
  if (b->max_feed) return fail(VADB200_E_STATE, "a ragged bank takes vadb200_stream_feed_ragged");
  if (!h->have_ffn) return fail(VADB200_E_STATE, "FFN weights not set (vadb200_set_ffn_weights)");
  if (reinterpret_cast<uintptr_t>(d_chunks) & 3) return fail(VADB200_E_INVALID, "chunks must be 4-byte aligned");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  BankParams bp;
  bp.n_streams = b->n; bp.hist = b->d_hist.get(); bp.ring = b->d_ring.get(); bp.fed = b->d_fed.get();
  bp.chunks = d_chunks; bp.labels = d_labels; bp.logits = d_logits;
  bp.tw1 = h->d_tw.get(); bp.tw2 = h->d_tw.get() + 256; bp.feat_mode = VADB200_FEAT_ANALYSER;
  bp.prev = b->d_prev.get();
  bp.fe = frontend_on(h) ? frontend_of(h) : FrontEnd{nullptr, 0.0f};
  const unsigned grid = (b->n + kStepFrames - 1) / kStepFrames;
  return launched(1, [&] {
    if (b->d_seg)  // speech on: every feed advances the segment state
      stream_feed_speech_kernel<StreamSeg><<<grid, kThreads, kStreamSmemBytes, st>>>(bp, h->par,
                                                                                    bank_seg(b, d_rows, d_bounds));
    else
      stream_feed_kernel<<<grid, kThreads, kStreamSmemBytes, st>>>(bp, h->par);
  });
}

}  // namespace

int vadb200_stream_bank_reset(vadb200_bank* b, void* stream) {
  if (!b) return fail(VADB200_E_INVALID, "bank is null");
  CU(cudaSetDevice(b->h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (b->max_feed) {
    CU(cudaMemsetAsync(b->d_pcm.get(), 0, static_cast<size_t>(b->n) * b->ring_len * sizeof(int16_t), st));
    CU(cudaMemsetAsync(b->d_total.get(), 0, static_cast<size_t>(b->n) * sizeof(long long), st));
  } else {
    CU(cudaMemsetAsync(b->d_hist.get(), 0, static_cast<size_t>(b->n) * 320 * sizeof(int16_t), st));
    CU(cudaMemsetAsync(b->d_fed.get(), 0, static_cast<size_t>(b->n) * sizeof(int), st));
    CU(cudaMemsetAsync(b->d_prev.get(), 0, static_cast<size_t>(b->n) * sizeof(int16_t), st));
  }
  CU(cudaMemsetAsync(b->d_ring.get(), 0, static_cast<size_t>(b->n) * 5 * kNCep * sizeof(float), st));
  if (b->d_seg) CU(cudaMemsetAsync(b->d_seg.get(), 0, b->seg_bytes, st));
  return 0;
}

int vadb200_stream_feed(vadb200_bank* b, const int16_t* d_chunks, uint8_t* d_labels, float* d_logits, void* stream) {
  return launch_stream_feed(b, d_chunks, d_labels, d_logits, nullptr, nullptr, stream);
}

int vadb200_stream_feed_ragged(vadb200_bank* b, const int16_t* d_samples, const int64_t* d_offsets, int32_t* d_counts,
                               uint8_t* d_labels, float* d_logits, uint8_t* d_rows, int64_t* d_bounds, void* stream) {
  if (!b || !d_samples || !d_offsets || !d_counts || !d_labels) return fail(VADB200_E_INVALID, "null argument");
  if (!b->max_feed) return fail(VADB200_E_STATE, "not a ragged bank (vadb200_stream_bank_create_ragged)");
  vadb200_handle* h = b->h;
  if (!h->have_ffn) return fail(VADB200_E_STATE, "FFN weights not set (vadb200_set_ffn_weights)");
  if ((d_rows || d_bounds) && !b->d_seg) return fail(VADB200_E_STATE, "speech is off (vadb200_stream_bank_set_speech)");
  if (reinterpret_cast<uintptr_t>(d_samples) & 1) return fail(VADB200_E_INVALID, "samples must be 2-byte aligned");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  RaggedParams rp;
  rp.n_streams = b->n; rp.max_feed = b->max_feed; rp.ring_len = b->ring_len; rp.max_rows = ragged_max_rows(b->max_feed);
  rp.pcm = b->d_pcm.get(); rp.total = b->d_total.get(); rp.ring = b->d_ring.get();
  rp.samples = d_samples; rp.offsets = reinterpret_cast<const long long*>(d_offsets);
  rp.counts = d_counts; rp.labels = d_labels; rp.logits = d_logits; rp.rows = d_rows; rp.bounds = d_bounds;
  rp.tw1 = h->d_tw.get(); rp.tw2 = h->d_tw.get() + 256; rp.feat_mode = VADB200_FEAT_ANALYSER;
  rp.fe = frontend_on(h) ? frontend_of(h) : FrontEnd{nullptr, 0.0f};
  const unsigned grid = (b->n + kStepFrames - 1) / kStepFrames;
  return launched(1, [&] {
    if (b->d_seg)  // speech on: every feed advances the segment state
      stream_ragged_speech_kernel<StreamSeg><<<grid, kThreads, kStreamSmemBytes, st>>>(rp, h->par,
                                                                                      bank_seg(b, nullptr, nullptr));
    else
      stream_ragged_kernel<<<grid, kThreads, kStreamSmemBytes, st>>>(rp, h->par);
  });
}

int vadb200_stream_bank_set_speech(vadb200_bank* b, int enable, int min_speech_rows, int min_silence_rows,
                                   int pad_rows, void* stream) {
  if (!b) return fail(VADB200_E_INVALID, "bank is null");
  if (enable) {
    for (int v : {min_speech_rows, min_silence_rows, pad_rows})
      if (v < 0 || v > kSpeechMaxParam) return fail(VADB200_E_INVALID, "speech parameters must lie in [0, 1000] rows");
  }
  CU(cudaSetDevice(b->h->device));
  CU(cudaFree(b->d_seg.release()));  // waits for work in flight that may still use it; reports its failure
  b->seg_bytes = 0;
  if (enable) {
    const SmoothParams sp = smooth_params(min_speech_rows, min_silence_rows, pad_rows);
    const int w1 = sp.G > 1 ? seg_ring_words(sp.G - 1) : 0, w2 = sp.S > 1 ? seg_ring_words(sp.S - 1) : 0;
    const size_t bytes = static_cast<size_t>(w1 + w2 + 2) * b->n * sizeof(uint32_t);
    CU(dev_alloc(b->d_seg, bytes));
    b->sp = sp;
    b->seg_bytes = bytes;
  }
  return vadb200_stream_bank_reset(b, stream);
}

int vadb200_stream_bank_speech_delay(const vadb200_bank* b) { return b && b->d_seg ? b->sp.H : -1; }

int vadb200_stream_feed_speech(vadb200_bank* b, const int16_t* d_chunks, uint8_t* d_labels, float* d_logits,
                               uint8_t* d_rows, int64_t* d_bounds, void* stream) {
  if (!b) return fail(VADB200_E_INVALID, "bank is null");
  if (!b->d_seg) return fail(VADB200_E_STATE, "speech is off (vadb200_stream_bank_set_speech)");
  return launch_stream_feed(b, d_chunks, d_labels, d_logits, d_rows, d_bounds, stream);
}

int vadb200_stream_bank_end_streams(vadb200_bank* b, const uint8_t* d_end, uint8_t* d_tail_rows,
                                    int64_t* d_tail_bounds, void* stream) {
  if (!b || !d_end) return fail(VADB200_E_INVALID, "null argument");
  CU(cudaSetDevice(b->h->device));
  const StreamSeg g = bank_seg(b, nullptr, nullptr);
  const int words = g.meta ? (g.d1 ? seg_ring_words(g.d1) : 0) + (g.d2 ? seg_ring_words(g.d2) : 0) : 0;
  const size_t smem = static_cast<size_t>(words) * kSegEndThreads * sizeof(uint32_t);
  const unsigned grid = (b->n + kSegEndThreads - 1) / kSegEndThreads;
  if (b->max_feed)
    return launched(1, [&] {
      stream_end_ragged_kernel<<<grid, kSegEndThreads, smem, static_cast<cudaStream_t>(stream)>>>(
          g, d_end, b->n, b->d_total.get(), b->d_ring.get(), g.meta ? d_tail_rows : nullptr,
          g.meta ? d_tail_bounds : nullptr);
    });
  return launched(1, [&] {
    stream_end_kernel<<<(b->n + kSegEndThreads - 1) / kSegEndThreads, kSegEndThreads, smem,
                        static_cast<cudaStream_t>(stream)>>>(g, d_end, b->n, b->d_hist.get(), b->d_ring.get(),
                                                             b->d_fed.get(), b->d_prev.get(),
                                                             g.meta ? d_tail_rows : nullptr,
                                                             g.meta ? d_tail_bounds : nullptr);
  });
}

#if defined(VADB_DEBUG_HOOKS)
// Occupancy experiment (hook build only, not in the public header): FFT phase alone at minb CTAs per SM.
int vadb200_exp_fft(vadb200_plan* p, const int16_t* d_pcm, int64_t pcm_len, int minb, void* stream) {
  vadb200_handle* h = p->h;
  CU(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  FusedParams fp = base_params(p);
  fp.pcm = d_pcm; fp.pcm_len = pcm_len; fp.seg_begin = 0; fp.seg_end = static_cast<int>(p->segs.size());
  fp.counter = p->d_counter.get() + 2 * (p->launch_seq.fetch_add(1) % kPlanCounters);
  const int grid = std::min<int>(fp.seg_end, minb * h->num_sms);
  const auto run = [&](auto kernel) {
    CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kExpSmemBytes));
    return launched(0, [&] { kernel<<<grid, kThreads, kExpSmemBytes, st>>>(fp, h->d_sink.get()); });
  };
  if (minb == 1) return run(exp_fft_kernel<1>);
  if (minb == 2) return run(exp_fft_kernel<2>);
  if (minb == 3) return run(exp_fft_kernel<3>);
  return run(exp_fft_kernel<4>);
}
#endif

// ---- FFN training (learning/ffn_trainer.py:104-175) --------------------------------------------------------
int vadb200_trainer_create(vadb200_handle* h, int64_t max_batch, float lr, float rho, float eps, vadb200_trainer** out) {
  if (!h || !out || max_batch < 1) return fail(VADB200_E_INVALID, "bad argument");
  *out = nullptr;
  CU(cudaSetDevice(h->device));
  std::unique_ptr<vadb200_trainer> t(new (std::nothrow) vadb200_trainer());
  if (!t) return fail(VADB200_E_NOMEM, "host allocation failed");
  t->h = h; t->device = h->device; t->max_batch = max_batch; t->lr = lr; t->rho = rho; t->eps = eps;
  const long long n_part = (max_batch + kTrainRows - 1) / kTrainRows;
  CU(dev_alloc(t->d_state, 3 * kNParams * sizeof(float)));
  CU(cudaMemset(t->d_state.get(), 0, 3 * kNParams * sizeof(float)));
  CU(dev_alloc(t->d_partial, n_part * (kNParams + 1) * sizeof(float)));
  CU(dev_alloc(t->d_loss, sizeof(float)));
  CU(cudaFuncSetAttribute(ffn_train_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTrain2SmemBytes));
  if (h->have_ffn)  // start from the handle's classifier
    CU(cudaMemcpy(t->d_state.get(), &h->par, kNParams * sizeof(float), cudaMemcpyHostToDevice));
  *out = t.release();
  return 0;
}

int vadb200_trainer_destroy(vadb200_trainer* t) {
  delete t;
  return 0;
}

int vadb200_trainer_set_weights(vadb200_trainer* t, const float* W1, const float* b1, const float* W2, const float* b2,
                                const float* W3, const float* b3, const float* W4, const float* b4, int reset_optimizer) {
  const float* src[8] = {W1, b1, W2, b2, W3, b3, W4, b4};
  if (!t || std::count(src, src + 8, nullptr)) return fail(VADB200_E_INVALID, "null argument");
  std::vector<float> v(kNParams);
  pack_params(src, v.data());
  CU(cudaSetDevice(t->h->device));
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(t->d_state.get(), v.data(), kNParams * sizeof(float), cudaMemcpyHostToDevice));
  if (reset_optimizer) CU(cudaMemset(t->d_state.get() + kNParams, 0, 2 * kNParams * sizeof(float)));
  return 0;
}

int vadb200_trainer_get_weights(vadb200_trainer* t, float* W1, float* b1, float* W2, float* b2, float* W3, float* b3,
                                float* W4, float* b4) {
  float* dst[8] = {W1, b1, W2, b2, W3, b3, W4, b4};
  if (!t || std::count(dst, dst + 8, nullptr)) return fail(VADB200_E_INVALID, "null argument");
  std::vector<float> v(kNParams);
  CU(cudaSetDevice(t->h->device));
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(v.data(), t->d_state.get(), kNParams * sizeof(float), cudaMemcpyDeviceToHost));
  unpack_params(v.data(), dst);
  return 0;
}

int vadb200_train_on_batch(vadb200_trainer* t, const float* d_x, const uint8_t* d_y, int64_t n, float* h_loss,
                           void* stream) {
  if (!t || n < 1 || !d_x || !d_y) return fail(VADB200_E_INVALID, "bad argument");
  if (n > t->max_batch) return fail(VADB200_E_INVALID, "batch larger than the trainer's max_batch");
  CU(cudaSetDevice(t->h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int n_tiles = static_cast<int>((n + kTrainRows - 1) / kTrainRows);
  const int n_part = std::min(n_tiles, t->h->num_sms);   // persistent CTAs: one partial gradient each
  float* state = t->d_state.get();
  const int rc = launched(2, [&] {
    ffn_train_grad_kernel<<<n_part, kTr2Threads, kTrain2SmemBytes, st>>>(state, d_x, d_y, n, 1.0f / static_cast<float>(n),
                                                                           t->d_partial.get());
    ffn_train_update_kernel<<<(kNParams + 1 + 255) / 256, 256, 0, st>>>(state, state + kNParams, state + 2 * kNParams,
                                                                         t->d_partial.get(), n_part, t->lr, t->rho,
                                                                         t->eps, t->d_loss.get());
  });
  if (rc) return rc;
  ++t->steps;
  if (h_loss) {
    CU(cudaMemcpyAsync(h_loss, t->d_loss.get(), sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  return 0;
}

// ---- bench support -----------------------------------------------------------------------------------------
int vadb200_synth_pcm(vadb200_handle* h, int16_t* d_out, int64_t n_utt, int64_t utt_samples, int64_t utt_stride,
                      uint32_t seed, int64_t first_utt, void* stream) {
  if (!h || !d_out || n_utt < 0 || utt_samples < 0 || utt_stride < utt_samples) return fail(VADB200_E_INVALID, "bad argument");
  if (n_utt == 0 || utt_samples == 0) return 0;
  CU(cudaSetDevice(h->device));
  const long long total = n_utt * utt_samples;
  const unsigned grid = static_cast<unsigned>(std::min<long long>((total + 255) / 256, 32ll * h->num_sms));
  return launched(1, [&] {
    synth_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_out, n_utt, utt_samples, utt_stride, seed,
                                                                      first_utt);
  });
}

int vadb200_fp32_peak(vadb200_handle* h, int variant, int iters, double* tflops_out) {
  if (!h || !tflops_out || iters < 1 || variant < 0 || variant > 6) return fail(VADB200_E_INVALID, "bad argument");
  CU(cudaSetDevice(h->device));
  Event e0, e1;
  CU(make_event(e0, cudaEventDefault));
  CU(make_event(e1, cudaEventDefault));
  const int grid = h->num_sms * 8;
  float* sink = h->d_sink.get();
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CU(cudaEventRecord(e0.get(), nullptr));
    const int rc = launched(1, [&] {
      if (variant == 0) fp32_peak_kernel<0><<<grid, 256>>>(sink, iters, 1.0000001f, 1e-9f);
      else if (variant == 1) fp32_peak_kernel<1><<<grid, 256>>>(sink, iters, 1.0000001f, 1e-9f);
      else if (variant == 2) fp32x2_peak_kernel<2><<<grid, 256>>>(sink, iters, 1.0000001f, 1e-9f);
      else if (variant == 3) fp32x2_peak_kernel<3><<<grid, 256>>>(sink, iters, 1.0000001f, 1e-9f);
      else if (variant == 4) fp32mix_peak_kernel<8><<<grid, 256>>>(sink, iters, 1.0000001f, 1e-9f);
      else if (variant == 5) fp32mix_peak_kernel<4><<<grid, 256>>>(sink, iters, 1.0000001f, 1e-9f);
      else fp32mix_peak_kernel<0><<<grid, 256>>>(sink, iters, 1.0000001f, 1e-9f);
    });
    if (rc) return rc;
    CU(cudaEventRecord(e1.get(), nullptr));
    CU(cudaEventSynchronize(e1.get()));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0.get(), e1.get()));
    const double per_rep = variant <= 1 ? 2.0 * 16 : variant <= 3 ? 4.0 * 16
                         : variant == 4 ? 4.0 * 8 + 2.0 * 8 : variant == 5 ? 4.0 * 8 + 2.0 * 4 : 4.0 * 8;
    const double flops = per_rep * 8 * static_cast<double>(iters) * 256.0 * grid;
    if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  *tflops_out = best;
  return 0;
}

// ---- speech segments (vad_segments.cuh) -----------------------------------------------------------------
namespace {
constexpr long long kWsAlign = 256;
long long ws_round(long long b) { return (b + kWsAlign - 1) / kWsAlign * kWsAlign; }
// workspace: tile counts int2[n_tiles] | tile prefixes longlong2[n_tiles + 1] | smoothed rows (when not asked)
struct SpeechWs {
  long long counts, prefix, smoothed, total;
};
SpeechWs speech_ws(const vadb200_plan* p) {
  SpeechWs w;
  const long long nt = static_cast<long long>(p->tiles.size());
  w.counts = 0;
  w.prefix = ws_round(nt * static_cast<long long>(sizeof(int2)));
  w.smoothed = w.prefix + ws_round((nt + 1) * static_cast<long long>(sizeof(longlong2)));
  w.total = w.smoothed + ws_round(p->total_rows);
  return w;
}
bool misaligned(const void* ptr, uintptr_t a) { return (reinterpret_cast<uintptr_t>(ptr) & (a - 1)) != 0; }
}  // namespace

int64_t vadb200_plan_max_speech_segments(const vadb200_plan* p) {
  if (!p || p->mode == VADB200_MODE_MFCC) return -1;
  return p->max_speech_segs;
}

int64_t vadb200_plan_speech_workspace_bytes(const vadb200_plan* p) {
  if (!p || p->mode == VADB200_MODE_MFCC) return -1;
  return speech_ws(p).total;
}

int vadb200_plan_speech_segments(vadb200_plan* p, const uint8_t* d_labels, int min_speech_rows, int min_silence_rows,
                                 int pad_rows, uint8_t* d_smoothed, int64_t* d_segments, int64_t* d_segment_offsets,
                                 int64_t* d_speech_offsets, void* d_workspace, int64_t workspace_bytes, void* stream) {
  if (!p) return fail(VADB200_E_INVALID, "plan is null");
  if (p->mode == VADB200_MODE_MFCC) return fail(VADB200_E_INVALID, "speech segments need a MODE_VAD or MODE_DATASET plan");
  for (int v : {min_speech_rows, min_silence_rows, pad_rows})
    if (v < 0 || v > kSpeechMaxParam) return fail(VADB200_E_INVALID, "row parameters must lie in [0, 1000]");
  const SpeechWs ws = speech_ws(p);
  if (!d_workspace || workspace_bytes < ws.total) return fail(VADB200_E_INVALID, "workspace is null or too small");
  if (misaligned(d_workspace, 16)) return fail(VADB200_E_INVALID, "workspace must be 16-byte aligned");
  if (!d_segment_offsets) return fail(VADB200_E_INVALID, "d_segment_offsets is null");
  if (p->total_rows > 0 && (!d_labels || !d_segments)) return fail(VADB200_E_INVALID, "d_labels / d_segments is null");
  if (misaligned(d_segments, 8) || misaligned(d_segment_offsets, 8) || misaligned(d_speech_offsets, 8))
    return fail(VADB200_E_INVALID, "segment and offset arrays must be 8-byte aligned");
  CU(cudaSetDevice(p->h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned char* wsb = static_cast<unsigned char*>(d_workspace);
  int2* counts = reinterpret_cast<int2*>(wsb + ws.counts);
  longlong2* prefix = reinterpret_cast<longlong2*>(wsb + ws.prefix);
  uint8_t* sm = d_smoothed ? d_smoothed : wsb + ws.smoothed;
  const int n_tiles = static_cast<int>(p->tiles.size());
  const SmoothParams sp = smooth_params(min_speech_rows, min_silence_rows, pad_rows);
  const long long utt_blocks = (p->n_utt + 1 + kSpeechThreads - 1) / kSpeechThreads;
  const unsigned grid = static_cast<unsigned>(std::max<long long>(n_tiles, utt_blocks));
  return launched(n_tiles > 0 ? 3 : 2, [&] {
    if (n_tiles > 0)
      speech_smooth_kernel<<<n_tiles, kSpeechThreads, smooth_smem_bytes(sp.H), st>>>(d_labels, p->d_tiles.get(),
                                                                                   p->d_row_off.get(), sp, sm, counts);
    speech_scan_kernel<<<1, kSpeechScanThreads, 0, st>>>(counts, n_tiles, prefix);
    speech_segments_kernel<<<grid, kSpeechThreads, 0, st>>>(
        sm, p->d_tiles.get(), p->d_row_off.get(), prefix, n_tiles, p->d_utt_tile.get(), p->n_utt,
        reinterpret_cast<long long*>(d_segments), reinterpret_cast<long long*>(d_segment_offsets),
        reinterpret_cast<long long*>(d_speech_offsets));
  });
}

int vadb200_plan_gather_speech(vadb200_plan* p, const int16_t* d_pcm, int64_t pcm_len, const int64_t* d_segments,
                               const int64_t* d_segment_offsets, const int64_t* d_speech_offsets, int16_t* d_out,
                               int64_t out_capacity, void* stream) {
  if (!p) return fail(VADB200_E_INVALID, "plan is null");
  if (p->mode == VADB200_MODE_MFCC) return fail(VADB200_E_INVALID, "speech segments need a MODE_VAD or MODE_DATASET plan");
  int rc = check_pcm(p, d_pcm, pcm_len);
  if (rc) return rc;
  if (out_capacity < 0) return fail(VADB200_E_INVALID, "out_capacity < 0");
  if (!d_segment_offsets || !d_speech_offsets) return fail(VADB200_E_INVALID, "offset arrays are null");
  if (p->total_rows > 0 && !d_segments) return fail(VADB200_E_INVALID, "d_segments is null");
  if (out_capacity > 0 && !d_out) return fail(VADB200_E_INVALID, "d_out is null");
  if (misaligned(d_out, 16)) return fail(VADB200_E_INVALID, "d_out must be 16-byte aligned");
  if (misaligned(d_segments, 8) || misaligned(d_segment_offsets, 8) || misaligned(d_speech_offsets, 8))
    return fail(VADB200_E_INVALID, "segment and offset arrays must be 8-byte aligned");
  if (p->total_rows == 0 || out_capacity == 0) return 0;
  CU(cudaSetDevice(p->h->device));
  // output hops are split evenly over a grid sized to keep HBM busy; CTAs past the speech exit at once
  const long long max_hops = p->total_rows;
  const unsigned grid = static_cast<unsigned>(std::max<long long>(1, std::min<long long>(8ll * p->h->num_sms, max_hops)));
  return launched(1, [&] {
    speech_gather_kernel<<<grid, kSpeechThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        d_pcm, p->d_pcm_off.get(), p->n_utt, reinterpret_cast<const long long*>(d_segments),
        reinterpret_cast<const long long*>(d_segment_offsets), reinterpret_cast<const long long*>(d_speech_offsets),
        d_out, out_capacity);
  });
}

// ---- other sample rates and formats (vad_resample.cuh) ----------------------------------------------------------
int vadb200_decode_pcm(vadb200_handle* h, const void* d_raw, int format, int channels, int big_endian,
                       const int64_t* d_src_start, const int64_t* d_dst_start, const int64_t* d_len, int n_seg,
                       int64_t max_len, float* d_dst, void* stream) {
  if (format < VADB200_PCM_S16 || format > VADB200_PCM_F64) return fail(VADB200_E_INVALID, "unknown sample format");
  if (channels < 1 || channels > kMaxChannels) return fail(VADB200_E_INVALID, "channels must be in [1, 32]");
  if (n_seg < 0 || max_len < 0) return fail(VADB200_E_INVALID, "bad argument");
  if (n_seg > 65535) return fail(VADB200_E_INVALID, "at most 65535 segments per call");
  const int align = format == VADB200_PCM_S24 ? 1 : kPcmBytes[format];
  if (misaligned(d_raw, align)) return fail(VADB200_E_INVALID, "raw stream must be aligned to the sample size");
  if (misaligned(d_dst, 4)) return fail(VADB200_E_INVALID, "d_dst must be 4-byte aligned");
  if (!h) return fail(VADB200_E_INVALID, "handle is null");
  if (n_seg == 0 || max_len == 0) return 0;
  if (!d_raw || !d_src_start || !d_dst_start || !d_len || !d_dst) return fail(VADB200_E_INVALID, "null argument");
  CU(cudaSetDevice(h->device));
  const unsigned gx = static_cast<unsigned>(std::min<long long>((max_len + 255) / 256, 4ll * h->num_sms));
  const dim3 grid(gx, static_cast<unsigned>(n_seg));
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  const uint8_t* raw = static_cast<const uint8_t*>(d_raw);
  const long long* src = reinterpret_cast<const long long*>(d_src_start);
  const long long* dst = reinterpret_cast<const long long*>(d_dst_start);
  const long long* len = reinterpret_cast<const long long*>(d_len);
  return launched(1, [&] { enqueue_decode_pcm(format, grid, st, raw, channels, big_endian, src, dst, len, d_dst); });
}

int64_t vadb200_resampled_length(int64_t n, int src_rate) {
  int up = 0, down = 0;
  if (n < 0 || !resample_ratio(src_rate, &up, &down)) return -1;
  return resampled_length(n, up, down);
}

int64_t vadb200_resample_taps(int src_rate, double* h_taps) {
  int up = 0, down = 0;
  if (!resample_ratio(src_rate, &up, &down)) return -1;
  const std::vector<double> taps = resample_taps(up, down);
  if (h_taps) std::memcpy(h_taps, taps.data(), taps.size() * sizeof(double));
  return static_cast<int64_t>(taps.size());
}

int vadb200_resampler_create(vadb200_handle* h, int src_rate, vadb200_resampler** out) {
  if (!out) return fail(VADB200_E_INVALID, "out is null");
  *out = nullptr;
  int up = 0, down = 0;
  if (!resample_ratio(src_rate, &up, &down))
    return fail(VADB200_E_UNSUPPORTED,
                "sample rate must be an integer in [4000, 384000] Hz with max(up, down) <= 1024 for 16000 Hz");
  if (!h) return fail(VADB200_E_INVALID, "handle is null");
  std::unique_ptr<vadb200_resampler> r(new (std::nothrow) vadb200_resampler());
  if (!r) return fail(VADB200_E_NOMEM, "host allocation failed");
  r->device = h->device;
  r->num_sms = h->num_sms;
  r->d = resample_design(up, down);
  CU(cudaSetDevice(h->device));
  int optin = 0;
  CU(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
  if (r->d.smem > static_cast<size_t>(optin)) return fail(VADB200_E_UNSUPPORTED, "resampler tile exceeds shared memory");
  // the largest opt-in for every resampler: one resampler's attribute never limits another's
  CU(resample_allow_smem(optin));
  const std::vector<float> taps = polyphase_taps(r->d, resample_taps(up, down));
  CU(dev_upload(r->d_taps, taps.data(), taps.size()));
  *out = r.release();
  return 0;
}

int vadb200_resampler_destroy(vadb200_resampler* r) {
  delete r;
  return 0;
}

int64_t vadb200_resample_workspace_bytes(const vadb200_resampler* r, int64_t n_utt) {
  if (!r || n_utt < 0) return -1;
  return std::max<int64_t>(n_utt, 1) * static_cast<int64_t>(sizeof(ResampleUtt));
}

int vadb200_resample_packed(vadb200_resampler* r, int in_format, const void* d_in, const int64_t* h_in_offsets,
                            const int64_t* h_in_lengths, int64_t n_utt, int16_t* d_out, int64_t out_capacity,
                            int64_t* h_out_offsets, void* d_workspace, int64_t workspace_bytes, void* stream) {
  if (!r) return fail(VADB200_E_INVALID, "resampler is null");
  if (in_format != VADB200_PCM_S16 && in_format != VADB200_PCM_F32)
    return fail(VADB200_E_INVALID, "in_format must be VADB200_PCM_S16 or VADB200_PCM_F32");
  if (n_utt < 0 || out_capacity < 0) return fail(VADB200_E_INVALID, "bad argument");
  if (!h_out_offsets || (n_utt > 0 && (!h_in_offsets || !h_in_lengths)))
    return fail(VADB200_E_INVALID, "null argument");
  if (misaligned(d_in, in_format == VADB200_PCM_S16 ? 2 : 4) || misaligned(d_out, 16) || misaligned(d_workspace, 16))
    return fail(VADB200_E_INVALID, "d_in must be aligned to its sample, d_out and the workspace to 16 bytes");
  if (n_utt > 0x7fffffffll) return fail(VADB200_E_INVALID, "too many utterances");
  const ResampleDesign& d = r->d;
  std::vector<ResampleUtt> utts(static_cast<size_t>(n_utt));
  long long out_pos = 0, tiles = 0;
  for (long long u = 0; u < n_utt; ++u) {
    const long long off = h_in_offsets[u], n = h_in_lengths[u];
    if (off < 0 || n < 0 || n > (1ll << 40)) return fail(VADB200_E_INVALID, "offsets and lengths must be >= 0");
    const long long m = resampled_length(n, d.up, d.down);
    utts[u] = ResampleUtt{off, n, out_pos, tiles};
    h_out_offsets[u] = out_pos;
    out_pos += (m + 7) / 8 * 8;
    tiles += (m + d.T - 1) / d.T;
  }
  h_out_offsets[n_utt] = out_pos;
  if (out_pos > out_capacity) return fail(VADB200_E_INVALID, "out_capacity is smaller than the resampled batch");
  if (tiles > 0x7fffffffll) return fail(VADB200_E_INVALID, "batch too large for one call");
  if (tiles == 0) return 0;
  if (!d_in || !d_out) return fail(VADB200_E_INVALID, "null argument");
  if (!d_workspace || workspace_bytes < vadb200_resample_workspace_bytes(r, n_utt))
    return fail(VADB200_E_INVALID, "workspace smaller than vadb200_resample_workspace_bytes");
  CU(cudaSetDevice(r->device));
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  ResampleUtt* ws = static_cast<ResampleUtt*>(d_workspace);
  const int n_fill = static_cast<int>((n_utt + kResampleFill - 1) / kResampleFill);
  ResampleParams a;
  a.in = d_in; a.out = d_out; a.utts = ws; a.n_utt = static_cast<int>(n_utt); a.taps = r->d_taps.get();
  a.up = d.up; a.down = d.down; a.half = d.half; a.K = d.K; a.Ks = d.Ks; a.q = d.q; a.H = d.H; a.win = d.win;
  a.taps_floats = (d.up * d.Ks + 3) / 4 * 4;
  return launched(n_fill + 1, [&] {
    enqueue_resample(in_format == VADB200_PCM_S16, a, utts.data(), n_utt, tiles, d.smem, st);
  });
}

}  // extern "C"
