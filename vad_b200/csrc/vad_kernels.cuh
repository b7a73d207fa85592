// vad_kernels.cuh -- sm_100a kernels of the fused MFCC + FFN VAD path.
//
// fused_kernel<MODE, TC>: persistent CTAs (2 per SM, 256 threads) pull *segments* (runs of
// consecutive frames of one utterance) from an atomic work counter.  Per 32-frame step:
//   1. PCM for the step (5360 int16 = 31 hops + one frame) arrives in shared memory by one
//      TMA bulk copy (cp.async.bulk + mbarrier), double-buffered one step ahead; overlapping
//      frames are re-read from shared memory, never from HBM.
//   2. FFT: each warp transforms 4 frames in ONE pass: a half-warp (16 threads) carries two
//      frames per thread as packed register pairs, so every butterfly / twiddle / split / power
//      operation is one FFMA2 / FADD2 / FMUL2 for both frames (sm_100a packed fp32):
//      pruned DFT16 -> twiddle -> 16x16 transpose in shared memory (re plane, then im plane)
//      -> DFT16 -> partner shuffle -> real-FFT split -> |X|^2 into the pair tile
//      [123 bin pairs + sink row][32 cols][2 bins] through per-thread base pointers (P2Store).
//   3. mel + log: lane = frame, warps 3-7 each own a run of consecutive filters and load every
//      power pair once (mel2_run); weights are uniform-register FFMA2 operands; exact-zero -> eps; log2.
//   4. DCT, one step behind: lane = frame, warps 0-3 transform two coefficient pairs per pass over
//      the 26 log-energies (folded DCT-II x lifter x log10(2) matrix); the result is a 64-bit element
//      of the 288-slot coefficient-pair MFCC ring in shared memory (carries the +-2 frame halo
//      across steps, so no frame is ever transformed twice inside a segment).
// The step has no CTA-wide bar.sync: two split-phase mbarriers ("P free", "P full", one arrival per
// warp) order the power tile; only block steps use CTA barriers.
// Block phase: MODE 0 / 1 flush MFCC / dataset rows (every 8 steps); MODE 2 builds the 5-frame window
// features and runs Dense 39-64-32-16-3 -- on FP32 CUDA cores (TC = 0, every 8 steps), as one tcgen05
// tile of 128 frames with TMEM accumulators (TC = 1, tf32 hi/lo operands, every 4 steps) or as two such
// tiles of 128 frames side by side in TMEM (TC = 2, fp16 hi/lo operands, every 8 steps) -- then
// argmax == VOICED, 1-byte label.
//
// Reference lines restated: mfcc.py:59-78; dataset/file_processing.py:47-70,99-101;
// realtime_analysis/sklearn_analyser.py:46-82,103-107; learning/ffn_trainer.py:104-116.
#pragma once

#include <cuda_runtime.h>

#include "vad_core.cuh"
#include "ffn_tc.cuh"

namespace vadb {

constexpr int kThreads = 256;
constexpr int kWarps = 8;
constexpr int kStepFrames = 32;
constexpr int kRing = 288;                                     // MFCC ring slots (modulus)
constexpr int kPPitch = 34;                                    // == 2 (mod 32): conflict-free P stores
constexpr int kStageSamples = (kStepFrames - 1) * kHop + kFrame;  // 5360
constexpr int kStagePad = 5376;                                // samples; 10752 B, 128-B multiple
constexpr int kBlockSteps = 8;                                 // block phase every 256 frames

constexpr int kOffPcm = 0;
constexpr int kOffExch = kOffPcm + 2 * kStagePad * 2;                       // 21504
constexpr int kOffP = kOffExch + kWarps * 2 * kExchFrame * 8;               // + 34816
constexpr int kP2Bytes = (kP2RowsAlloc * kP2Pitch * 4 + 15) & ~15;          // pair tile: 123 rows x 66 floats + sink row
constexpr int kOffLogE = kOffP + kP2Bytes;                                  // + 32480
constexpr int kLogEFloats = kNMel * 32;                                     // one step's log-mel tile
constexpr int kOffRing = kOffLogE + 2 * kLogEFloats * 4;                    // + 6656 (two tiles: the DCT runs one step behind)
constexpr int kOffTw1 = kOffRing + ((kRingRows * ring_pitch(kRing) * 4 + 15) & ~15);  // + 16192: coefficient-pair rows
constexpr int kOffTw2 = kOffTw1 + 256 * 8;
constexpr int kOffBar = kOffTw2 + 128 * 8;
constexpr int kOffSeg = kOffBar + 48;                                       // 6 mbarriers: pcm x2, weights, mma, P free, P full
constexpr int kFusedSmemBytes = kOffSeg + 16;                               // s_seg, s_tmem
constexpr int kBlockStepsTc = 4;                                            // tf32 tensor-core FFN: one M=128 tile
// A block phase reads the window of centres out_done .. computed - 3, i.e. up to kBlockSteps * 32 + 4 ring slots back.
static_assert(kBlockSteps * kStepFrames + 4 <= kRing, "the MFCC ring must hold a whole block phase's windows");
static_assert(kTcBlobBytes <= kWarps * 2 * kExchFrame * 8 + kP2Bytes, "weight blob must fit exch + P");
static_assert(kBlockSteps * kStepFrames * kNFeat * 4 + 16 <= kWarps * 2 * kExchFrame * 8 + kP2Bytes,
              "dataset-row staging tile must fit exch + P");
static_assert(2 * (kFusedSmemBytes + 1024) <= 233472, "two CTAs per SM");

struct Segment {
  long long pcm_start;  // sample index of the first frame's first sample (multiple of 8)
  long long out_start;  // first output row of the segment
  int n_frames;         // MFCC frames to compute (outputs + 4 in window modes)
  int cont;             // 1: the segment continues an utterance (the sample before it is real), 0: utterance start
};

// Opt-in front end of the fused kernels' fused_fe_kernel variant (vadb200_set_frontend): pre-emphasis coefficient and
// the handle's window table (vad_core.cuh fft_load_pcm2_fe; all ones when no window is set).
struct FrontEnd {
  const cf2* win;
  float preemph;
};

// Timing-experiment hooks (phase ablation mask, clock64 stamps) are compiled in only with
// -DVADB_DEBUG_HOOKS (tools/ab.sh builds); the product build has none of their branches.
#if defined(VADB_DEBUG_HOOKS)
#define VADB_DBG(p) ((p).debug_skip)
#else
#define VADB_DBG(p) 0
#endif

struct FusedParams {
  const int16_t* pcm;
  long long pcm_len;      // one past the last readable sample index (relative to pcm)
  const Segment* segs;
  int seg_begin, seg_end;
  int* counter;           // counter[0]: next segment, counter[1]: CTAs finished (the last one resets both)
  const cf2* tw1;
  const cf2* tw2;
  uint8_t* labels;
  float* logits;
  float* feats;
  float* rows;
  long long row_base;     // subtracted from Segment::out_start (chunked host runs)
  int feat_mode;
  const unsigned char* tc_blob;  // canonical hi/lo tf32 weight blob (ffn_tc.cuh), TC variant only
  long long* dbg_ts;             // timing experiments only: clock64 stamps of CTA 0's block phases [n][16]
  int debug_skip;                // timing experiments only (env VADB200_DEBUG_SKIP): 1 FFT, 2 mel, 4 DCT, 8 block phase,
                                 // 256 no second fp16 tile (tools/ablate.sh lists the rest)
};

// ---- PTX wrappers: mbarrier + TMA bulk copy (UBLKCP) --------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {  // release.cta
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// One arrival per warp: the __syncwarp orders the other lanes' shared-memory accesses before lane 0's release.
__device__ __forceinline__ void warp_arrive(uint64_t* bar, int lane) {
  __syncwarp();
  if (lane == 0) mbar_arrive(bar);
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

struct ShflXchg {
  int lane;
  __device__ __forceinline__ float operator()(float mine, int, bool, int partner) const {
    return __shfl_sync(0xffffffffu, mine, (lane & 16) | partner);
  }
  __device__ __forceinline__ f2 operator()(f2 mine, int, bool, int partner) const {
    const int src = (lane & 16) | partner;
    return mk2(__shfl_sync(0xffffffffu, mine.x, src), __shfl_sync(0xffffffffu, mine.y, src));
  }
};

// Four frames of a warp through the FFT: half-warp h = lanes 16h..16h+15, two frames per thread.
// ex: this half-warp's transpose scratch (kExchFrame 64-bit slots).
// store(bin, v): receives |2X|^2 of power bin `bin` for frame A (v.x) and frame B (v.y).
// before_store() runs after the second DFT16 and before the first power value is stored (the fused kernels put the
// CTA barrier that protects the previous step's power tile there: by then every warp has long left its mel phase).
// load(t, xr, xi) fills thread t's inputs (fft_load_pcm2 or, with the front end, fft_load_pcm2_fe).
template <int NZ, class LOAD, class PRE, class STORE>
__device__ __forceinline__ void warp_fft_quad(LOAD&& load, f2* ex, const cf2* s_tw1, const cf2* s_tw2, int lane,
                                               PRE&& before_store, STORE&& store) {
  const int t = lane & 15;
  f2 xr[16], xi[16];
  load(t, xr, xi);
  fft_pass1<NZ>(xr, xi, s_tw1, t);
  exch_store_plane(ex, t, xr);
  __syncwarp();
  exch_load_plane(ex, t, xr);
  __syncwarp();
  exch_store_plane(ex, t, xi);
  __syncwarp();
  exch_load_plane(ex, t, xi);
  __syncwarp();
  dft16<16>(xr, xi);
  before_store();
  fft_split_store(xr, xi, t, s_tw2, ShflXchg{lane}, store);
}
// The fused kernels' power tile: pair rows (bins 2q, 2q+1 side by side per column, vad_core.cuh p2_index); bins
// below the first mel bin are dropped.  Columns col (frame A) and col + 1 (frame B).
// Thread k1 of a half-warp stores bins k1 + 16 k2 ("lo") and 256 - k1 - 16 k2 ("hi"), k2 = 0 .. 7, plus bin 128 on
// thread 0.  In the pair tile both families are affine in k2 (+- 8 pair rows per step), so four per-thread pointers
// computed once per kernel replace all per-store index arithmetic.  Row kP2Rows ("bin 256") is a write-only sink:
// bins below the first mel bin (k2 == 0, k1 < 10), thread 0's bin 256 and the other threads' "bin 128" go there, which
// makes every store unconditional.
struct P2Store {
  static constexpr bool kHasSink = true;
  float* lo_base;   // bin k1
  float* hi_base;   // bin 256 - k1
  float* lo0;       // bin k1 if it is kept, else the sink
  float* mid_ptr;   // bin 128 (thread 0) or the sink
  __device__ __forceinline__ P2Store(float* P2, int col, int k1) {
    lo_base = P2 + p2_index(k1, col);              // may point below the tile for k1 < 10: only used with k2 >= 1
    hi_base = P2 + p2_index(256 - k1, col);
    // every lane of a warp gets its own word of the sink row (k1 + 16 h, h = half-warp = bit 3 of the column):
    // several lanes storing to one address would be serialised
    float* sink = P2 + kP2Rows * kP2Pitch + k1 + 2 * (col & 8);
    lo0 = k1 >= kMelFirstBin ? lo_base : sink;
    mid_ptr = k1 == 0 ? P2 + p2_index(128, col) : sink;
  }
  static __device__ __forceinline__ void put(float* q, f2 v) {
    q[0] = v.x;
    q[2] = v.y;
  }
  template <class K> __device__ __forceinline__ void lo(K, f2 v) const {
    constexpr int k2 = K::value;
    if constexpr (k2 == 0) put(lo0, v);
    else put(lo_base + 8 * k2 * kP2Pitch, v);
  }
  template <class K> __device__ __forceinline__ void hi(K, f2 v) const { put(hi_base - 8 * K::value * kP2Pitch, v); }
  __device__ __forceinline__ void mid(f2 v) const { put(mid_ptr, v); }
};

// Both frames of a warp (lanes 0-15 / 16-31) through the FFT; P column = frame slot fi.
template <int NZ, class LOAD>
__device__ __forceinline__ void warp_fft_pair(LOAD&& load, cf2* ex, const cf2* s_tw1, const cf2* s_tw2,
                                               float* s_P, int fi, int lane) {
  const int t = lane & 15;
  float xr[16], xi[16];
  load(xr, xi);
  fft_pass1<NZ>(xr, xi, s_tw1, t);
  exch_store(ex, t, xr, xi);
  __syncwarp();
  exch_load(ex, t, xr, xi);
  __syncwarp();
  dft16<16>(xr, xi);
  fft_split_store(xr, xi, t, s_tw2, ShflXchg{lane}, [&](int bin, float v) { s_P[bin * kPPitch + fi] = v; });
}

// Coalesced store of `total` consecutive floats starting at dst: a scalar head up to the first 16-byte
// boundary, 128-bit stores, scalar tail.  gen(j, v, cnt) produces elements j .. j + cnt - 1 (cnt <= 4).
template <int NTHREADS = kThreads, class GEN>
__device__ __forceinline__ void flush_flat(float* dst, int total, int tid, GEN&& gen) {
  if (total <= 0) return;
  const int head = min(total, static_cast<int>((16u - (reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u) >> 2);
  const int nq = (total - head) >> 2;
  for (int q = tid; q < nq; q += NTHREADS) {
    float v[4];
    gen(head + 4 * q, v, 4);
    *reinterpret_cast<float4*>(dst + head + 4 * q) = make_float4(v[0], v[1], v[2], v[3]);
  }
  const int tail0 = head + 4 * nq;
  if (tid < 2) {  // thread 0: head, thread 1: tail (each < 4 elements)
    const int j0 = tid == 0 ? 0 : tail0, cnt = tid == 0 ? head : total - tail0;
    if (cnt > 0) {
      float v[4];
      gen(j0, v, cnt);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i < cnt) dst[j0 + i] = v[i];
    }
  }
}

// One output row per thread: window features -> FFN -> decision (block phase / windows API).
// th: decision threshold (decide); 0 = argmax.
__device__ __forceinline__ void classify_row(const FfnParams& w, const float (&r)[5][kNCep], int feat_mode,
                                             uint8_t* labels, float* logits, float* feats, long long row, float th) {
  float x[kNFeat];
  const bool ok = window_features(r, feat_mode, x);
  float logit[kNCls];
  ffn_forward(w, x, logit);
  uint8_t lab = decide(logit, th);
  if (!ok) {
    logit[0] = logit[1] = logit[2] = NAN;
    lab = 0;
  }
  if (labels) labels[row] = lab;
  if (logits) {
    logits[row * 3 + 0] = logit[0];
    logits[row * 3 + 1] = logit[1];
    logits[row * 3 + 2] = logit[2];
  }
  if (feats) {
#pragma unroll
    for (int i = 0; i < kNFeat; ++i) feats[row * kNFeat + i] = x[i];
  }
}

// MODE 0: MFCC rows [T][13]; 1: dataset rows [T-5][39]; 2: VAD labels [T-5].
// TC (MODE 2 only): 0 = FFN on FP32 CUDA cores, 1 = FFN on tcgen05 kind::tf32 (hi/lo split, TMEM accumulators),
// 2 = tcgen05 kind::f16 on statically scaled fp16 hi/lo operands (half the MMAs, half the weight blob).
// FFN argument of the kernel variant: nothing (MFCC / dataset rows), the full FP32 weights, or the biases
// only (tensor-core FFN: the weights are the per-handle tcgen05 operand blob in global memory).
template <int MODE, int TC> struct FfnArgOf { using type = FfnNone; };
template <> struct FfnArgOf<2, 0> { using type = FfnParams; };
template <> struct FfnArgOf<2, 1> { using type = FfnBias; };
template <> struct FfnArgOf<2, 2> { using type = FfnBias; };

// The decision of the VAD block phase: argmax, or with the front-end variant the handle's threshold.
template <bool FE, class A>
__device__ __forceinline__ uint8_t decide_of(const float (&logit)[kNCls], const A& ffn) {
  if constexpr (FE && !std::is_same<A, FfnNone>::value) return decide(logit, ffn.thresh);
  else return decide(logit);
}

// FE: the front-end variant (fused_fe_kernel).  Its PCM stage starts kStageOffFe samples into each buffer and the
// sample before the step's first frame sits just below it (0 at an utterance start), so fft_load_pcm2_fe finds
// every frame's previous sample at word -1.  The step's 5360 samples + 8 still fit the 5376-sample buffer.
constexpr int kStageOffFe = 8;
static_assert(kStageSamples + kStageOffFe <= kStagePad, "front-end stage offset must fit the PCM buffer");

// tid comes from the kernel: threadIdx.x read inside the kernel carries the launch bound's range (0 .. 255), which the
// code generation relies on (read here, the default kernels' SASS would change).
template <int MODE, int TC, bool FE>
__device__ __forceinline__ void fused_body(const FusedParams& p, const typename FfnArgOf<MODE, TC>::type& ffn,
                                           const FrontEnd& fe, const int tid) {
  static_assert(TC == 0 || MODE == 2, "tensor-core FFN only exists in VAD mode");
  constexpr int kBlk = TC == 1 ? kBlockStepsTc : kBlockSteps;
  constexpr int kStageOff = FE ? kStageOffFe : 0;
  extern __shared__ __align__(128) unsigned char smem[];
  int16_t* s_pcm = reinterpret_cast<int16_t*>(smem + kOffPcm);
  cf2* s_exch = reinterpret_cast<cf2*>(smem + kOffExch);
  float* s_P = reinterpret_cast<float*>(smem + kOffP);
  float* s_logE = reinterpret_cast<float*>(smem + kOffLogE);
  float* s_ring = reinterpret_cast<float*>(smem + kOffRing);
  cf2* s_tw1 = reinterpret_cast<cf2*>(smem + kOffTw1);
  cf2* s_tw2 = reinterpret_cast<cf2*>(smem + kOffTw2);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + kOffBar);
  int* s_seg = reinterpret_cast<int*>(smem + kOffSeg);

  const int warp = tid >> 5, lane = tid & 31, h = lane >> 4, t = lane & 15;

  s_tw1[tid] = p.tw1[tid];
  if (tid < 128) s_tw2[tid] = p.tw2[tid];
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + kOffSeg + 8);
  if (tid == 0) {
    mbar_init(&s_bar[0], 1);
    mbar_init(&s_bar[1], 1);
    mbar_init(&s_bar[2], 1);
    mbar_init(&s_bar[3], 1);
    mbar_init(&s_bar[4], kWarps);  // "P free": every warp has finished the mel of the previous step
    mbar_init(&s_bar[5], kWarps);  // "P full": every warp has stored its power columns of this step
    fence_mbar_init();
  }
  uint32_t tm_base = 0, w_par = 0, mma_par = 0;
  int dbg_n = 0;
  if (TC) {
    if (warp == 0) tmem_alloc(s_tmem, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tm_base = *s_tmem;
  }

  unsigned gstep = 0;  // loads issued so far by this CTA == steps started; buffer = gstep & 1
  Segment seg{};
  const P2Store p2store(s_P, col_of_halfwarp(warp, h), t);  // this thread's power-store pointers, fixed for the kernel
  __syncthreads();                 // mbarrier inits visible
  warp_arrive(&s_bar[4], lane);    // the power tile starts out free

  // (Staggering the block-phase schedule of the two CTAs sharing an SM -- per-SM arrival rank via
  // %smid -- was tried against the lockstep hypothesis and measured neutral: 232.1 vs 231.1 ms.  Strict
  // turn-taking of the FFT phases between the two CTAs through a per-SM word in global memory, so that one
  // CTA's FFT always overlaps the other's mel / DCT / classifier, was 3.3x SLOWER: 696 vs 212 ms.  Letting the warps
  // whose frame slots lie past the segment end skip the transform of a short last step: 214.7 vs 212.0 ms.)

  // Called by warp 0 only (the bulk copy is issued by thread 0, the < 8-sample tail is copied by lanes 0-6).
  auto issue_load = [&](int step, int buf) {
    const long long start = seg.pcm_start + static_cast<long long>(step) * (kStepFrames * kHop);
    const long long avail = p.pcm_len - start;
    const int nsmp = avail >= kStageSamples ? kStageSamples : (avail > 0 ? static_cast<int>(avail) : 0);
    const int bulk = (nsmp * 2) & ~15;
    int16_t* dst = s_pcm + buf * kStagePad + kStageOff;
    if (tid == 0) {
      mbar_arrive_expect_tx(&s_bar[buf], static_cast<uint32_t>(bulk));
      if (bulk) bulk_g2s(dst, p.pcm + start, static_cast<uint32_t>(bulk), &s_bar[buf]);
    }
    const int tail0 = bulk >> 1;  // < 8 samples past the last whole 16-byte chunk of the buffer
    if (tid < nsmp - tail0) dst[tail0 + tid] = p.pcm[start + tail0 + tid];
    // the previous sample: part of the utterance unless this is the first step of an utterance's first segment
    // (published like the tail samples: by warp 0's arrival on "P full" / the barrier after the first load)
    if (FE && tid == 31) dst[-1] = (step > 0 || seg.cont) ? p.pcm[start - 1] : int16_t(0);
  };

  for (;;) {
    __syncthreads();
    if (tid == 0) *s_seg = p.seg_begin + atomicAdd(p.counter, 1);
    __syncthreads();
    const int si = *s_seg;
    if (si >= p.seg_end) break;
    seg = p.segs[si];
    const int n = seg.n_frames;
    const int nsteps = (n + kStepFrames - 1) / kStepFrames;
    int out_done = (MODE == 0) ? 0 : 2;
    bool dct_pending = false;  // the previous step's log-mel tile still waits for its DCT
    if (nsteps > 0 && warp == 0) issue_load(0, gstep & 1);
    __syncthreads();

    for (int s = 0; s < nsteps; ++s, ++gstep) {
      const int buf = gstep & 1;
      if (s + 1 < nsteps && warp == 0) issue_load(s + 1, buf ^ 1);
      mbar_wait(&s_bar[buf], (gstep >> 1) & 1);

      // Two split-phase barriers (mbarrier arrive / wait, one arrival per warp) replace CTA-wide bar.syncs, so a warp
      // only ever waits for data it needs and the warps of a CTA drift apart instead of marching in lockstep:
      //   s_bar[4] "P free": arrive after the mel of step s - 1, wait before the first power store of step s
      //                      (by then the arrivals are ~ one FFT old);
      //   s_bar[5] "P full": arrive after the last power store, wait before the mel; the DCT of step s - 1 sits
      //                      between the two, it needs nothing from this step.
      // Both complete once per step: parity = gstep & 1.
      const uint32_t par = gstep & 1;
      auto dct_step = [&](int sd) {
        if (!(VADB_DBG(p) & 4)) {
          const float* le = s_logE + (sd & 1) * kLogEFloats + lane;
          const int col = (sd * kStepFrames + slot_of_col(lane)) % kRing;  // lane = P column
          // Warps 0-3 share the transform, so a column's 26 log-energies are loaded 4 times instead of 7: warps 0-2
          // take two coefficient pairs each, warp 3 the seventh; the mel runs (tools/gen_tables.py) are sized so that
          // these warps carry little or no mel work.
          if (warp < 3) {
            float ra, rb, rc, rd;
            dct_coef4<32>(le, 2 * warp, ra, rb, rc, rd);
            *reinterpret_cast<float2*>(s_ring + ring_idx(4 * warp, col, kRing)) = make_float2(ra, rb);
            *reinterpret_cast<float2*>(s_ring + ring_idx(4 * warp + 2, col, kRing)) = make_float2(rc, rd);
          } else if (warp == 3) {
            float ra, rb;
            dct_coef2<32>(le, 6, ra, rb);
            s_ring[ring_idx(12, col, kRing)] = ra;
          }
        }
      };

      // ---- FFT phase ---------------------------------------------------------------------
      const uint32_t* stage32 = reinterpret_cast<const uint32_t*>(s_pcm + buf * kStagePad + kStageOff);
      if (!(VADB_DBG(p) & 1)) {
        // half-warp h: frame slots 4 warp + h and + 2 (PCM 80 words apart per slot -> the two half-warps
        // read different banks), P columns 4 warp + 2 h, + 1
        f2* ex = reinterpret_cast<f2*>(s_exch) + (warp * 2 + h) * kExchFrame;
        const uint32_t* w32a = stage32 + (warp * 4 + h) * (kHop / 2);
        warp_fft_quad<13>(
            [&](int tt, f2 (&xr)[16], f2 (&xi)[16]) {
              if constexpr (FE) fft_load_pcm2_fe(w32a, kHop, tt, fe.preemph, fe.win, xr, xi);
              else fft_load_pcm2(w32a, kHop, tt, xr, xi);
            },
            ex, s_tw1, s_tw2, lane, [&] { mbar_wait(&s_bar[4], par); }, p2store);
      } else {
        mbar_wait(&s_bar[4], par);
      }
      warp_arrive(&s_bar[5], lane);

      // ---- DCT -> MFCC ring, one step behind ---------------------------------------------------
      // The log-mel tile of step s - 1 is complete (every warp arrived on "P free" after its mel).
      if (dct_pending) dct_step(s - 1);
      mbar_wait(&s_bar[5], par);

      // ---- mel + log phase -----------------------------------------------------------------
      // (a rolled, table-driven mel loop -- one small code body for all warps, weights in shared memory -- was
      // measured 5.8 % slower than these eight straight-line regions: its loads are latency-exposed)
      if (!(VADB_DBG(p) & 2))
        mel2_run_dispatch<kP2Pitch, 32>(warp, s_P + 2 * lane, s_logE + (s & 1) * kLogEFloats + lane);
      warp_arrive(&s_bar[4], lane);
      const int computed = min((s + 1) * kStepFrames, n);
      const bool block_now = (((s + 1) % kBlk) == 0 || s == nsteps - 1) && !(VADB_DBG(p) & 8);
      const bool tc_now = TC && block_now && (computed - 2 - out_done) > 0;  // block-uniform
      dct_pending = !block_now;

      // A step that is followed by a block phase transforms its own log-mel tile right away, behind a CTA barrier.
      if (block_now) {
        if (tc_now) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // exch/P generic accesses before the TMA overwrite
        __syncthreads();
        if (tc_now && tid == 0 && !(VADB_DBG(p) & 16)) {  // exch + P are idle until the next FFT phase: land the weight blob during the DCT
          constexpr uint32_t blob_bytes = TC == 2 ? kTc16BlobBytes : kTcBlobBytes;
          mbar_arrive_expect_tx(&s_bar[2], blob_bytes);
          bulk_g2s(smem + kOffExch, p.tc_blob, blob_bytes, &s_bar[2]);
        }
        dct_step(s);
      }

      if (block_now) {
        __syncthreads();
        if (MODE == 0) {
          // rows are contiguous in global memory: flat float index j <-> (frame j / 13, coefficient j % 13)
          float* dst = p.rows + (seg.out_start - p.row_base + out_done) * kNCep;
          const int first = out_done;
          flush_flat(dst, (computed - out_done) * kNCep, tid, [&](int j, float (&v)[4], int cnt) {
            int fr = j / kNCep, cf = j - fr * kNCep;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              if (i < cnt) v[i] = s_ring[ring_idx(cf, (first + fr) % kRing, kRing)];
              if (++cf == kNCep) { cf = 0; ++fr; }
            }
          });
          out_done = computed;
        } else if (MODE == 1) {
          // Dataset rows [c (13) | d1 (13) | d2 (13)] of centres out_done .. computed - 3 (<= 256): thread = centre
          // builds its 39 values with the packed window arithmetic and writes them into a staging tile that has the
          // layout of the output rows (exch + P are idle here; a row is 39 floats = 7 banks apart: conflict free);
          // the tile then leaves with 128-bit coalesced stores, without any per-element index arithmetic.
          const int n_valid = computed - 2 - out_done;
          if (n_valid > 0) {  // block-uniform
            float* dst = p.rows + (seg.out_start - p.row_base + (out_done - 2)) * kNFeat;
            // staging starts at the same offset within 16 bytes as dst, so 128-bit chunks line up on both sides
            float* stage = reinterpret_cast<float*>(smem + kOffExch) + ((reinterpret_cast<uintptr_t>(dst) & 15u) >> 2);
            if (tid < n_valid) {
              float xa[24], xb[24];
              window_features_pairs<0, 4, kRing, 24>(s_ring, out_done + tid, 1, xa);
              window_features_pairs<4, 7, kRing, 24>(s_ring, out_done + tid, 1, xb);
              float* row = stage + tid * kNFeat;
#pragma unroll
              for (int g = 0; g < 3; ++g) {
#pragma unroll
                for (int k = 0; k < 8; ++k) row[g * kNCep + k] = xa[6 * (k >> 1) + 2 * g + (k & 1)];
#pragma unroll
                for (int k = 0; k < 5; ++k) row[g * kNCep + 8 + k] = xb[6 * (k >> 1) + 2 * g + (k & 1)];
              }
            }
            __syncthreads();
            flush_flat(dst, n_valid * kNFeat, tid, [&](int j, float (&v)[4], int cnt) {
              if (cnt == 4) {
                const float4 q = *reinterpret_cast<const float4*>(stage + j);
                v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
              } else {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                  if (i < cnt) v[i] = stage[j + i];
              }
            });
            __syncthreads();  // the next FFT phase rewrites exch / P
          }
          out_done = max(out_done, computed - 2);
        } else if (!TC) {
          const int c = out_done + tid;
          if (c <= computed - 3) {
            float r[5][kNCep];
#pragma unroll
            for (int d = 0; d < 5; ++d) {
              const int col = (c - 2 + d) % kRing;
#pragma unroll
              for (int k = 0; k < kNCep; ++k) r[d][k] = s_ring[ring_idx(k, col, kRing)];
            }
            if constexpr (MODE == 2 && TC == 0)
              classify_row(ffn, r, p.feat_mode, p.labels, p.logits, p.feats, seg.out_start - p.row_base + (c - 2),
                           FE ? ffn.thresh : 0.0f);
          }
          out_done = max(out_done, computed - 2);
        } else if constexpr (TC == 2) {
          // ---- fp16 tensor-core FFN: two M = 128 tiles, thread = frame = TMEM lane of tile warp / 4 ---------------
          const int n_valid = computed - 2 - out_done;  // centres out_done .. computed-3 (<= 256)
          if (n_valid > 0) {                            // block-uniform (== tc_now)
            long long* ts = nullptr;
#if defined(VADB_DEBUG_HOOKS)
            if (p.dbg_ts && blockIdx.x == 0 && tid == 0 && dbg_n < 64) ts = p.dbg_ts + 16 * dbg_n;
#endif
            if (ts) ts[0] = clock64();
            const bool valid = tid < n_valid;
            const int c = out_done + (valid ? tid : 0);
            const long long row = seg.out_start - p.row_base + (c - 2);
            const uint32_t tl = ffn_tc16_tile2_lane(tm_base, warp);
            // The frame's 48 layer-1 columns, one 24-column half (coefficient pairs 0-3, then 4-6) at a time.  Validity
            // stays in a register: ReLU's fmaxf swallows NaNs, so it cannot be read back from the logits.
            bool ok = true;
#pragma unroll
            for (int hidx = 0; hidx < 2; ++hidx) {
              float xl[24];
              if (VADB_DBG(p) & 64) {
#pragma unroll
                for (int i = 0; i < 24; ++i) xl[i] = 0.5f;
              } else {
                ok = (hidx == 0 ? window_features_pairs<0, 4, kRing, 24>(s_ring, c, p.feat_mode, xl)
                                : window_features_pairs<4, 7, kRing, 24>(s_ring, c, p.feat_mode, xl)) && ok;
              }
              tc16_store_a1_half(tl, hidx, xl);
              if (p.feats && valid) {
                const int k0 = hidx ? 8 : 0, nk = hidx ? 5 : 8;  // xl[6 (k / 2) + 2 g + k % 2], k relative to k0
#pragma unroll
                for (int k = 0; k < 8; ++k)
#pragma unroll
                  for (int g = 0; g < 3; ++g)
                    if (k < nk) p.feats[row * kNFeat + g * kNCep + k0 + k] = xl[6 * (k >> 1) + 2 * g + (k & 1)];
              }
            }
            if (ts) ts[1] = clock64();
            if (!(VADB_DBG(p) & 16)) mbar_wait(&s_bar[2], w_par);  // weight blob landed (issued before the DCT phase)
            if (ts) ts[2] = clock64();
            float logit[kNCls];
            // tile 1 only when it holds a valid centre (hook build: mask 256 never issues it, to time one chain)
            const bool two_tiles = n_valid > 128 && !(VADB_DBG(p) & 256);
            mma_par = ffn_tc16_tile2(ffn, logit, tm_base, warp, two_tiles, tid == 0, smem_u32(smem + kOffExch), &s_bar[3],
                                     mma_par, ts);
            ++dbg_n;
            if (valid) {
              uint8_t lab = decide_of<FE>(logit, ffn);  // logits are in registers: no TMEM round trip
              if (!ok) {
                logit[0] = logit[1] = logit[2] = NAN;
                lab = 0;
              }
              p.labels[row] = lab;
              if (p.logits) {
                p.logits[row * 3 + 0] = logit[0];
                p.logits[row * 3 + 1] = logit[1];
                p.logits[row * 3 + 2] = logit[2];
              }
            }
            if (!(VADB_DBG(p) & 16)) w_par ^= 1u;
            __syncthreads();  // MMAs done reading the blob before the next FFT phase rewrites exch / P
          }
          out_done = max(out_done, computed - 2);
        } else {
          // ---- tf32 tensor-core FFN: one M = 128 tile over all 8 warps ------------------------------
          const int n_valid = computed - 2 - out_done;  // centres out_done .. computed-3 (<= 128)
          if (n_valid > 0) {                            // block-uniform (== tc_now)
            unsigned char* wdst = smem + kOffExch;
            {
              // thread (warp % 4, lane) = frame = TMEM lane; the two threads sharing a frame (hidx = warp / 4)
              // build the features of cepstral coefficients 0-6 / 7-12 and split every layer's columns.
              const int fr = tid & 127, hidx = tid >> 7;
              long long* ts = nullptr;
#if defined(VADB_DEBUG_HOOKS)
              if (p.dbg_ts && blockIdx.x == 0 && tid == 0 && dbg_n < 64) ts = p.dbg_ts + 16 * dbg_n;
#endif
              if (ts) ts[0] = clock64();
              const bool valid = fr < n_valid;
              const int c = out_done + (valid ? fr : 0);
              const uint32_t tl = tm_base + (static_cast<uint32_t>(32 * (warp & 3)) << 16);
              float xl[24], logit[kNCls];
              // the half's validity flag travels through shared memory (logE is idle here): ReLU's fmaxf
              // swallows NaNs, so validity cannot be read back from the logits
              bool ok_half = true;
              if (VADB_DBG(p) & 64) {
#pragma unroll
                for (int i = 0; i < 24; ++i) xl[i] = 0.5f;
              } else {
                ok_half = (hidx == 0) ? window_features_pairs<0, 4, kRing, 24>(s_ring, c, p.feat_mode, xl)
                                      : window_features_pairs<4, 7, kRing, 24>(s_ring, c, p.feat_mode, xl);
              }
              s_logE[tid] = ok_half ? 1.0f : 0.0f;
              if (ts) ts[1] = clock64();
              tc_store_a1_half(tl, hidx, xl);
              if (p.feats && valid) {
                const long long row = seg.out_start - p.row_base + (c - 2);
                const int k0 = hidx ? 8 : 0, nk = hidx ? 5 : 8;  // xl[6 (k / 2) + 2 g + k % 2], k relative to k0
#pragma unroll
                for (int k = 0; k < 8; ++k)
#pragma unroll
                  for (int g = 0; g < 3; ++g)
                    if (k < nk) p.feats[row * kNFeat + g * kNCep + k0 + k] = xl[6 * (k >> 1) + 2 * g + (k & 1)];
              }
              if (!(VADB_DBG(p) & 16)) mbar_wait(&s_bar[2], w_par);  // weight blob landed (issued before the DCT phase)
              if (ts) ts[2] = clock64();
              if constexpr (TC == 1)
                mma_par = ffn_tc_tile<2>(ffn, logit, tm_base, warp & 3, hidx, tid == 0, smem_u32(wdst), &s_bar[3], mma_par,
                                         ts, VADB_DBG(p));
              ++dbg_n;
              if (valid && hidx == 0) {
                const bool ok = s_logE[fr] != 0.0f && s_logE[128 + fr] != 0.0f;  // ordered by the tile's bar.syncs
                uint8_t lab = decide_of<FE>(logit, ffn);  // logits are in registers: no TMEM round trip
                if (!ok) {
                  logit[0] = logit[1] = logit[2] = NAN;
                  lab = 0;
                }
                const long long row = seg.out_start - p.row_base + (c - 2);
                p.labels[row] = lab;
                if (p.logits) {
                  p.logits[row * 3 + 0] = logit[0];
                  p.logits[row * 3 + 1] = logit[1];
                  p.logits[row * 3 + 2] = logit[2];
                }
              }
            }
            if (!(VADB_DBG(p) & 16)) w_par ^= 1u;
            __syncthreads();  // MMAs done reading the blob before the next FFT phase rewrites exch / P
          }
          out_done = max(out_done, computed - 2);
        }
      }
    }
  }
  if (TC) {
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm_base, kTmemCols);
  }
  // Every CTA reaches this point only after the work counter ran past seg_end, so the last one to
  // arrive can re-arm the counter pair for the plan's next launch (no memset between launches).
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(p.counter + 1, 1) == static_cast<int>(gridDim.x) - 1) {
      p.counter[0] = 0;
      p.counter[1] = 0;
      __threadfence();
    }
  }
}

template <int MODE, int TC>
__global__ void __launch_bounds__(kThreads, 2) fused_kernel(const __grid_constant__ FusedParams p,
                                                            const __grid_constant__ typename FfnArgOf<MODE, TC>::type ffn) {
  fused_body<MODE, TC, false>(p, ffn, FrontEnd{nullptr, 0.0f}, threadIdx.x);
}
// The same kernel with the opt-in front end and decision threshold; launched only when the handle sets either, so the
// default path above keeps its code.
template <int MODE, int TC>
__global__ void __launch_bounds__(kThreads, 2) fused_fe_kernel(const __grid_constant__ FusedParams p,
                                                               const __grid_constant__ typename FfnArgOf<MODE, TC>::type ffn,
                                                               const __grid_constant__ FrontEnd fe) {
  fused_body<MODE, TC, true>(p, ffn, fe, threadIdx.x);
}

// Stand-alone tensor-core FFN over feature rows [n][39] (classifier.predict duck type): one CTA =
// one 128-row tile.  Same tile routines as the fused kernel's block phase.  The fp16 scales hold only for
// features within the kFeatBound* of their group, which caller rows need not be: with KIND 2 a tile holding
// any row beyond them runs on the tf32 blob instead (fp16 would overflow to inf and return NaN logits).
constexpr int kFfnTcSmemBytes = kTcBlobBytes + 64;
template <int KIND>  // 1: tf32 operands, 2: fp16 operands where the tile's rows allow
__global__ void __launch_bounds__(128) ffn_tc_rows_kernel(const float* x, long long n, const unsigned char* blob16,
                                                          const unsigned char* blob32, uint8_t* labels, float* logits,
                                                          const __grid_constant__ FfnBias fb) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kTcBlobBytes);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + kTcBlobBytes + 32);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(s_tmem, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm_base = *s_tmem;
  if (KIND == 1 && tid == 0) {
    mbar_arrive_expect_tx(&bars[0], kTcBlobBytes);
    bulk_g2s(smem, blob32, kTcBlobBytes, &bars[0]);
  }
  const long long i = static_cast<long long>(blockIdx.x) * 128 + tid;
  const long long src = i < n ? i : n - 1;
  float v[kNFeat], logit[kNCls];
  bool ok = true, wide = false;
#pragma unroll
  for (int k = 0; k < kNFeat; ++k) {
    v[k] = x[src * kNFeat + k];
    ok = ok && (fabsf(v[k]) <= 3.0e38f);
    if constexpr (KIND == 2)
      wide = wide || fabsf(v[k]) > (k < kNCep ? kFeatBoundZ : k < 2 * kNCep ? kFeatBoundD1 : kFeatBoundD2);
  }
  bool fp16 = false;
  if constexpr (KIND == 2) {
    fp16 = !__syncthreads_or(wide);
    if (tid == 0) {
      const uint32_t bytes = fp16 ? kTc16BlobBytes : kTcBlobBytes;
      mbar_arrive_expect_tx(&bars[0], bytes);
      bulk_g2s(smem, fp16 ? blob16 : blob32, bytes, &bars[0]);
    }
  }
  mbar_wait(&bars[0], 0);
  {
    const uint32_t tl = tm_base + (static_cast<uint32_t>(32 * warp) << 16);
    float h0[24], h1[24];
#pragma unroll
    for (int i = 0; i < 24; ++i) h0[i] = h1[i] = 0.0f;
#pragma unroll
    for (int f = 0; f < kNFeat; ++f) {
      const int col = tc_feat_col(f);
      if (col < 24) h0[col] = v[f];
      else h1[col - 24] = v[f];
    }
    if (fp16) {
      tc16_store_a1_half(tl, 0, h0);
      tc16_store_a1_half(tl, 1, h1);
    } else {
      tc_store_a1_half(tl, 0, h0);
      tc_store_a1_half(tl, 1, h1);
    }
  }
  if (fp16) ffn_tc16_tile<1>(fb, logit, tm_base, warp, 0, tid == 0, smem_u32(smem), &bars[1], 0);
  else ffn_tc_tile<1>(fb, logit, tm_base, warp, 0, tid == 0, smem_u32(smem), &bars[1], 0);
  if (i < n) {
    uint8_t lab = decide(logit, fb.thresh);
    if (!ok) {
      logit[0] = logit[1] = logit[2] = NAN;
      lab = 0;
    }
    if (labels) labels[i] = lab;
    if (logits) {
      logits[i * 3 + 0] = logit[0];
      logits[i * 3 + 1] = logit[1];
      logits[i * 3 + 2] = logit[2];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tm_base, kTmemCols);
}

#if defined(VADB_DEBUG_HOOKS)
// Occupancy experiment (hook build only): the fused kernel's PCM staging + FFT phase with the power
// values folded into a per-thread checksum instead of the shared P tile, so the CTA needs only the
// PCM buffers + transpose scratch (59 KB) and 3-4 CTAs fit per SM.  MINB = min blocks per SM.
constexpr int kExpSmemBytes = 2 * kStagePad * 2 + kWarps * 2 * kExchFrame * 8 + 384 * 8 + 64;
template <int MINB>
__global__ void __launch_bounds__(kThreads, MINB) exp_fft_kernel(const FusedParams p, float* sink) {
  extern __shared__ __align__(128) unsigned char smem[];
  int16_t* s_pcm = reinterpret_cast<int16_t*>(smem);
  cf2* s_exch = reinterpret_cast<cf2*>(smem + 2 * kStagePad * 2);
  cf2* s_tw1 = reinterpret_cast<cf2*>(smem + 2 * kStagePad * 2 + kWarps * 2 * kExchFrame * 8);
  cf2* s_tw2 = s_tw1 + 256;
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_tw2 + 128);
  int* s_seg = reinterpret_cast<int*>(s_bar + 4);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, h = lane >> 4, t = lane & 15;
  s_tw1[tid] = p.tw1[tid];
  if (tid < 128) s_tw2[tid] = p.tw2[tid];
  if (tid == 0) {
    mbar_init(&s_bar[0], 1);
    mbar_init(&s_bar[1], 1);
    fence_mbar_init();
  }
  unsigned gstep = 0;
  float acc = 0.0f;
  Segment seg;
  auto issue_load = [&](int step, int buf) {
    const long long start = seg.pcm_start + static_cast<long long>(step) * (kStepFrames * kHop);
    const long long avail = p.pcm_len - start;
    const int nsmp = avail >= kStageSamples ? kStageSamples : (avail > 0 ? static_cast<int>(avail) : 0);
    const int bulk = (nsmp * 2) & ~15;
    if (tid == 0) {
      mbar_arrive_expect_tx(&s_bar[buf], static_cast<uint32_t>(bulk));
      if (bulk) bulk_g2s(s_pcm + buf * kStagePad, p.pcm + start, static_cast<uint32_t>(bulk), &s_bar[buf]);
    }
  };
  for (;;) {
    __syncthreads();
    if (tid == 0) *s_seg = p.seg_begin + atomicAdd(p.counter, 1);
    __syncthreads();
    const int si = *s_seg;
    if (si >= p.seg_end) break;
    seg = p.segs[si];
    const int nsteps = (seg.n_frames + kStepFrames - 1) / kStepFrames;
    issue_load(0, gstep & 1);
    __syncthreads();
    for (int s = 0; s < nsteps; ++s, ++gstep) {
      const int buf = gstep & 1;
      if (s + 1 < nsteps) issue_load(s + 1, buf ^ 1);
      mbar_wait(&s_bar[buf], (gstep >> 1) & 1);
      const uint32_t* stage32 = reinterpret_cast<const uint32_t*>(s_pcm + buf * kStagePad);
      cf2* ex = s_exch + (warp * 2 + h) * kExchFrame;
#pragma unroll 1
      for (int r = 0; r < 2; ++r) {
        const int fi = warp * 4 + r * 2 + h;
        const uint32_t* w32 = stage32 + fi * (kHop / 2);
        float xr[16], xi[16];
        fft_load_pcm(w32, t, xr, xi);
        fft_pass1<13>(xr, xi, s_tw1, t);
        exch_store(ex, t, xr, xi);
        __syncwarp();
        exch_load(ex, t, xr, xi);
        __syncwarp();
        dft16<16>(xr, xi);
        fft_split_store(xr, xi, t, s_tw2, ShflXchg{lane}, [&](int bin, float v) { acc = fmaf(v, 1e-12f * bin, acc); });
      }
      __syncthreads();  // the PCM buffer is re-filled two steps later
    }
  }
  if (acc == 123.456f) sink[0] = acc;
}
#endif

// ---- per-frame API kernels (explicit float32 frames; mfcc.py:59-78 one frame at a time) ----------
// One CTA = 32 frames (same step structure; frames read straight from global memory).
// what: 0 -> spectrum [n][256] (get_spec_mag), 1 -> MFCC [n][13] (get_mfcc).
constexpr int kFramesSmemBytes = kWarps * 2 * kExchFrame * 8 + kBins * kPPitch * 4 + kNMel * 32 * 4 + 384 * 8;

// fe: the handle's front end (fe.win == nullptr: none).
__global__ void __launch_bounds__(kThreads) frames_kernel(const float* frames, long long n, int frame_len, int what,
                                                         float* out, const cf2* tw1, const cf2* tw2, FrontEnd fe) {
  extern __shared__ __align__(128) unsigned char smem[];
  cf2* s_exch = reinterpret_cast<cf2*>(smem);
  float* s_P = reinterpret_cast<float*>(smem + kWarps * 2 * kExchFrame * 8);
  float* s_logE = s_P + kBins * kPPitch;
  cf2* s_tw1 = reinterpret_cast<cf2*>(s_logE + kNMel * 32);
  cf2* s_tw2 = s_tw1 + 256;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, h = lane >> 4, t = lane & 15;
  s_tw1[tid] = tw1[tid];
  if (tid < 128) s_tw2[tid] = tw2[tid];
  __syncthreads();
  const long long f0 = static_cast<long long>(blockIdx.x) * kStepFrames;
  cf2* ex = s_exch + (warp * 2 + h) * kExchFrame;
#pragma unroll 1
  for (int r = 0; r < 2; ++r) {
    const int fi = warp * 4 + r * 2 + h;
    const long long f = min(f0 + fi, n - 1);  // clamp: surplus slots recompute the last frame
    const float* fr = frames + f * frame_len;
    warp_fft_pair<16>(
        [&](float (&xr)[16], float (&xi)[16]) {
          if (fe.win) fft_load_f32_fe(fr, frame_len, t, fe.preemph, fe.win, xr, xi);
          else fft_load_f32(fr, frame_len, t, xr, xi);
        },
        ex, s_tw1, s_tw2, s_P, fi, lane);
  }
  __syncthreads();
  if (what == 0) {
    // |X/512|^2 = |2X|^2 * 2^-20
    for (int j = tid; j < kStepFrames * kBins; j += kThreads) {
      const int fi = j >> 8, k = j & 255;
      if (f0 + fi < n) out[(f0 + fi) * kBins + k] = s_P[k * kPPitch + fi] * 9.5367431640625e-07f;
    }
    return;
  }
  mel_group_dispatch<kPPitch, 32>(warp, s_P + lane, s_logE + lane);
  __syncthreads();
  if (f0 + lane < n) {
    out[(f0 + lane) * kNCep + warp] = dct_coef<32>(s_logE + lane, warp);
    if (warp + 8 < kNCep) out[(f0 + lane) * kNCep + warp + 8] = dct_coef<32>(s_logE + lane, warp + 8);
  }
}

// get_mfcc_from_spec (mfcc.py:72-78) for given spectra [n][256]: P = spec * 2^20 feeds the same
// mel / log / DCT code.  One CTA = 32 spectra.
__global__ void __launch_bounds__(kThreads) spec_to_mfcc_kernel(const float* spec, long long n, float* out) {
  __shared__ float s_P[kBins * kPPitch];
  __shared__ float s_logE[kNMel * 32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long f0 = static_cast<long long>(blockIdx.x) * kStepFrames;
  for (int j = tid; j < kStepFrames * kBins; j += kThreads) {
    const int fi = j >> 8, k = j & 255;
    const long long f = min(f0 + fi, n - 1);
    s_P[k * kPPitch + fi] = spec[f * kBins + k] * 1048576.0f;
  }
  __syncthreads();
  mel_group_dispatch<kPPitch, 32>(warp, s_P + lane, s_logE + lane);
  __syncthreads();
  if (f0 + lane < n) {
    out[(f0 + lane) * kNCep + warp] = dct_coef<32>(s_logE + lane, warp);
    if (warp + 8 < kNCep) out[(f0 + lane) * kNCep + warp + 8] = dct_coef<32>(s_logE + lane, warp + 8);
  }
}

// 5-frame MFCC windows [n][5][13] -> features / logits / labels (one thread per window).
__global__ void __launch_bounds__(128) windows_kernel(const float* win, long long n, int feat_mode, uint8_t* labels,
                                                      float* logits, float* feats, const __grid_constant__ FfnParams w) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float r[5][kNCep];
#pragma unroll
  for (int d = 0; d < 5; ++d)
#pragma unroll
    for (int k = 0; k < kNCep; ++k) r[d][k] = win[(i * 5 + d) * kNCep + k];
  classify_row(w, r, feat_mode, labels, logits, feats, i, w.thresh);
}

// classifier.predict duck type (sklearn_analyser.py:71): rows [n][39] -> class {0,1}, logits.
__global__ void __launch_bounds__(128) ffn_rows_kernel(const float* x, long long n, uint8_t* labels, float* logits,
                                                       const __grid_constant__ FfnParams w) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v[kNFeat];
  bool ok = true;
#pragma unroll
  for (int k = 0; k < kNFeat; ++k) {
    v[k] = x[i * kNFeat + k];
    ok = ok && (fabsf(v[k]) <= 3.0e38f);
  }
  float logit[kNCls];
  ffn_forward(w, v, logit);
  uint8_t lab = decide(logit, w.thresh);
  if (!ok) {
    logit[0] = logit[1] = logit[2] = NAN;
    lab = 0;
  }
  if (labels) labels[i] = lab;
  if (logits) {
    logits[i * 3 + 0] = logit[0];
    logits[i * 3 + 1] = logit[1];
    logits[i * 3 + 2] = logit[2];
  }
}

// mfcc.get_deltas (mfcc.py:81-82: a - b) and mfcc.lifter (mfcc.py:85-93) for standalone callers.
// op 0: out = a - b;  op 1: out[i] = a[i] * (1 + (L/2) sin(pi (i % ncoef) / L))  (L <= 0: copy).
__global__ void elementwise_kernel(int op, const float* a, const float* b, long long n, int ncoef, int L, float* out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (op == 0) {
    out[i] = a[i] - b[i];
  } else {
    const int k = static_cast<int>(i % ncoef);
    const float lift = (L > 0) ? 1.0f + (0.5f * L) * sinpif(static_cast<float>(k) / static_cast<float>(L)) : 1.0f;
    out[i] = lift * a[i];
  }
}

// ---- streaming bank (SKLearnAnalyzer.feed_frame for many streams, one 160-sample chunk each) -----
// State per stream (struct-of-arrays, stream fastest): hist int16[320], ring float[5][13] (slot 4 =
// newest), fed int32 (chunks fed so far).  Chunk j completes frame j-2 = hist[0:320] ++ chunk[0:80].
// Reference timing (sklearn_analyser.py:46-82): feeding frame i first classifies frame i-3 from the
// ring holding frames i-5..i-1, then pushes frame i.
struct BankParams {
  int n_streams;
  int16_t* hist;   // [n_streams][320]
  float* ring;     // [5*13][n_streams]
  int* fed;        // [n_streams]
  const int16_t* chunks;  // [n_streams][160]
  uint8_t* labels;
  float* logits;
  const cf2* tw1;
  const cf2* tw2;
  int feat_mode;
  int16_t* prev;          // [n_streams] the raw sample before the 320-sample history (front end only)
  FrontEnd fe;            // fe.win == nullptr: no front end
};
constexpr int kStreamFramePitch = 480;  // samples per staged row: [history 320 | chunk 160] (240 words == 16 mod 32)
constexpr int kStreamPBytes = kP2Bytes > (kNFeat + kH1 + kH2 + kH3 + kNCep) * 32 * 4
                                  ? kP2Bytes : (kNFeat + kH1 + kH2 + kH3 + kNCep) * 32 * 4;  // P tile, later activations
constexpr int kStreamRowsOff = 16;      // bytes below staged row 0: its word -1 (front end)
constexpr int kStreamSmemBytes = kStreamRowsOff + kStepFrames * kStreamFramePitch * 2 + kWarps * 2 * kExchFrame * 8 +
                                 kStreamPBytes + kNMel * 32 * 4 + 384 * 8;

// One CTA = 32 streams.  FFT: the fused kernel's packed two-frames-per-thread pass.  The decision
// tail is spread over all 8 warps with lane = stream: warp w owns cepstral coefficients w, w + 8
// (DCT, ring push, window features) and then 8 / 4 / 2 neurons of layers 1 / 2 / 3, activations
// handed over through shared memory (the idle P tile); weights are uniform constant-bank operands.
// SEG: the speech variant (stream_feed_speech_kernel) also runs each stream's online smoothing step
// (vad_segments.cuh seg_step, found when the variant is instantiated with Seg = StreamSeg) on the label warp 0
// holds, and writes the finalised row and its bound.
template <bool SEG, class Seg>
__device__ __forceinline__ void stream_feed_body(const BankParams& p, const FfnParams& w, const Seg& sg,
                                                 const int tid) {
  extern __shared__ __align__(128) unsigned char smem[];
  int16_t* s_fr = reinterpret_cast<int16_t*>(smem + kStreamRowsOff);
  cf2* s_exch = reinterpret_cast<cf2*>(smem + kStreamRowsOff + kStepFrames * kStreamFramePitch * 2);
  float* s_P = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(s_exch) + kWarps * 2 * kExchFrame * 8);
  float* s_logE = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(s_P) + kStreamPBytes);
  cf2* s_tw1 = reinterpret_cast<cf2*>(s_logE + kNMel * 32);
  cf2* s_tw2 = s_tw1 + 256;
  // after the mel phase the P tile is dead: activations live there
  float* s_x = s_P;                    // [39][32]
  float* s_h1 = s_x + kNFeat * 32;     // [64][32]
  float* s_h2 = s_h1 + kH1 * 32;       // [32][32]
  float* s_h3 = s_h2 + kH2 * 32;       // [16][32]
  int* s_ok = reinterpret_cast<int*>(s_h3 + kH3 * 32);  // [13][32]
  const int warp = tid >> 5, lane = tid & 31, h = lane >> 4;
  const int s0 = blockIdx.x * kStepFrames;
  s_tw1[tid] = p.tw1[tid];
  if (tid < 128) s_tw2[tid] = p.tw2[tid];
  // stage [hist 320 | chunk 160] per stream: every chunk sample is read exactly once (the chunks may live in
  // pinned host memory: zero-copy ticks), then roll the history in global memory from the staged copy
  for (int j = tid; j < kStepFrames * 240; j += kThreads) {  // 32-bit words: 160 hist + 80 chunk per stream
    const int fi = j / 240, wd = j - fi * 240;
    const int st = min(s0 + fi, p.n_streams - 1);
    const uint32_t v = (wd < 160) ? reinterpret_cast<const uint32_t*>(p.hist + static_cast<long long>(st) * 320)[wd]
                                  : reinterpret_cast<const uint32_t*>(p.chunks + static_cast<long long>(st) * 160)[wd - 160];
    reinterpret_cast<uint32_t*>(s_fr + fi * kStreamFramePitch)[wd] = v;
  }
  __syncthreads();
  // new history = old hist[160:320] ++ chunk[0:160] = staged words 80 .. 239
  for (int j = tid; j < kStepFrames * 160; j += kThreads) {
    const int fi = j / 160, wd = j - fi * 160;
    const int st = s0 + fi;
    if (st < p.n_streams)
      reinterpret_cast<uint32_t*>(p.hist + static_cast<long long>(st) * 320)[wd] =
          reinterpret_cast<const uint32_t*>(s_fr + fi * kStreamFramePitch)[80 + wd];
  }
  if (p.fe.win) {
    // Front end: a stream is one signal from its last reset.  The sample before the history goes to the high half of
    // the row's word -1 (the previous row's last chunk word: the roll above has consumed it), and the stream's new
    // previous sample is old hist[159], the one before the new history.
    __syncthreads();
    if (tid < kStepFrames) {
      int16_t* row = s_fr + tid * kStreamFramePitch;
      const int st = min(s0 + tid, p.n_streams - 1);
      row[-1] = p.prev[st];
      if (s0 + tid < p.n_streams) p.prev[st] = row[159];
    }
    __syncthreads();
  }
  {
    f2* ex = reinterpret_cast<f2*>(s_exch) + (warp * 2 + h) * kExchFrame;
    const uint32_t* w32 = reinterpret_cast<const uint32_t*>(s_fr + (warp * 4 + h) * kStreamFramePitch);
    warp_fft_quad<13>(
        [&](int t, f2 (&xr)[16], f2 (&xi)[16]) {
          if (p.fe.win) fft_load_pcm2_fe(w32, kStreamFramePitch, t, p.fe.preemph, p.fe.win, xr, xi);
          else fft_load_pcm2(w32, kStreamFramePitch, t, xr, xi);
        },
        ex, s_tw1, s_tw2, lane, [] {}, P2Store(s_P, col_of_halfwarp(warp, h), lane & 15));
  }
  __syncthreads();
  mel2_run_dispatch<kP2Pitch, 32>(warp, s_P + 2 * lane, s_logE + lane);
  __syncthreads();
  // ---- DCT + ring + window features: warp = coefficient (w, w + 8), lane = P column ----------------
  const int slot = slot_of_col(lane);      // stream of this lane inside the CTA
  const int st = s0 + slot;
  const bool live = st < p.n_streams;
  const long long ns = p.n_streams;
  const int fed = live ? p.fed[st] : 0;    // chunks fed before this one
  const int frame = fed - 2;               // index of the frame completed by this chunk (< 0: none yet)
  // (a row is classified once frame >= 5: the ring then holds frames frame-5 .. frame-1 and frame-3 is the centre)
#pragma unroll
  for (int rep = 0; rep < 2; ++rep) {
    const int k = warp + 8 * rep;
    if (k < kNCep) {                       // warp-uniform
      const float cnew = dct_coef<32>(s_logE + lane, k);
      float r[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
      if (live && frame >= 0) {
#pragma unroll
        for (int d = 0; d < 5; ++d) r[d] = p.ring[(d * kNCep + k) * ns + st];
#pragma unroll
        for (int d = 0; d < 4; ++d) p.ring[(d * kNCep + k) * ns + st] = r[d + 1];
        p.ring[(4 * kNCep + k) * ns + st] = cnew;
      }
      float z = r[2];
      bool ok = true;
      if (p.feat_mode == 0) {
        const float mu = mul_rn((((r[0] + r[1]) + r[2]) + r[3]) + r[4], 0.2f);   // as window_features
        const float d0 = r[0] - mu, d1 = r[1] - mu, d2 = r[2] - mu, d3 = r[3] - mu, d4 = r[4] - mu;
        const float var = fmaf(d4, d4, fmaf(d3, d3, fmaf(d2, d2, fmaf(d1, d1, d0 * d0)))) * 0.2f;
        const bool alleq = (r[0] == r[1]) && (r[1] == r[2]) && (r[2] == r[3]) && (r[3] == r[4]);
        z = alleq ? NAN : mul_rn(d2, vadb_rsqrt(var));
        ok = fabsf(z) <= 3.0e38f;
      }
      s_x[k * 32 + slot] = z;
      s_x[(kNCep + k) * 32 + slot] = r[3] - r[1];
      s_x[(2 * kNCep + k) * 32 + slot] = (r[4] - z) - (z - r[0]);
      s_ok[k * 32 + slot] = ok ? 1 : 0;
    }
  }
  __syncthreads();
  // ---- FFN, lane = stream (slot order from here on) --------------------------------------------------
  {
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = w.b1[8 * warp + j];
#pragma unroll 3
    for (int i = 0; i < kNFeat; ++i) {
      const float xv = s_x[i * 32 + lane];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(xv, w.W1[i * kH1 + 8 * warp + j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) s_h1[(8 * warp + j) * 32 + lane] = fmaxf(acc[j], 0.0f);
  }
  __syncthreads();
  {
    float acc[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[j] = w.b2[4 * warp + j];
#pragma unroll 4
    for (int i = 0; i < kH1; ++i) {
      const float a = s_h1[i * 32 + lane];
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j] = fmaf(a, w.W2[i * kH2 + 4 * warp + j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) s_h2[(4 * warp + j) * 32 + lane] = fmaxf(acc[j], 0.0f);
  }
  __syncthreads();
  {
    float acc[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) acc[j] = w.b3[2 * warp + j];
#pragma unroll 4
    for (int i = 0; i < kH2; ++i) {
      const float a = s_h2[i * 32 + lane];
#pragma unroll
      for (int j = 0; j < 2; ++j) acc[j] = fmaf(a, w.W3[i * kH3 + 2 * warp + j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) s_h3[(2 * warp + j) * 32 + lane] = fmaxf(acc[j], 0.0f);
  }
  __syncthreads();
  if (warp == 0) {
    const int stl = s0 + lane;
    if (stl < p.n_streams) {
      const int fedl = p.fed[stl];
      uint8_t lab = 255;
      float lg[3] = {NAN, NAN, NAN};
      if (fedl - 2 >= 5) {
        float acc[kNCls];
#pragma unroll
        for (int o = 0; o < kNCls; ++o) acc[o] = w.b4[o];
#pragma unroll
        for (int i = 0; i < kH3; ++i) {
          const float a = s_h3[i * 32 + lane];
#pragma unroll
          for (int o = 0; o < kNCls; ++o) acc[o] = fmaf(a, w.W4[i * kNCls + o], acc[o]);
        }
        bool ok = true;
#pragma unroll
        for (int k = 0; k < kNCep; ++k) ok = ok && (s_ok[k * 32 + lane] != 0);
        lab = decide(acc, w.thresh);
        if (ok) {
          lg[0] = acc[0]; lg[1] = acc[1]; lg[2] = acc[2];
        } else {
          lab = 0;
        }
      }
      p.fed[stl] = fedl + 1;
      p.labels[stl] = lab;
      if (p.logits) {
        p.logits[stl * 3 + 0] = lg[0];
        p.logits[stl * 3 + 1] = lg[1];
        p.logits[stl * 3 + 2] = lg[2];
      }
      if constexpr (SEG) {  // row fedl - 7 of the stream is this label
        uint8_t row = 255;
        long long bound = -1;
        if (lab != 255) seg_step(sg, stl, fedl - 7, lab != 0, row, bound);
        if (sg.rows) sg.rows[stl] = row;
        if (sg.bounds) sg.bounds[stl] = bound;
      }
    }
  }
}

__global__ void __launch_bounds__(kThreads) stream_feed_kernel(const BankParams p, const __grid_constant__ FfnParams w) {
  stream_feed_body<false>(p, w, 0, threadIdx.x);
}
// The same tick plus the bank's segment step (vadb200_stream_bank_set_speech); the plain kernel above keeps its code.
template <class Seg>
__global__ void __launch_bounds__(kThreads) stream_feed_speech_kernel(const BankParams p,
                                                                     const __grid_constant__ FfnParams w,
                                                                     const __grid_constant__ Seg sg) {
  stream_feed_body<true>(p, w, sg, threadIdx.x);
}

// ---- feature sink: scale_features (dataset/utils.py:5-32) on packed dataset rows [n][39] ----------------
// One scalar mean and one population standard deviation per group g in {mfcc, d1, d2} over all n x 13
// values of the step, float64 accumulation like numpy.  Three passes over the rows:
//   pass 0: acc[g] += sum v;   pass 1: acc[3 + g] += sum (v - mean_g)^2;   pass 2: v = (v - mean_g) / std_g.
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
__global__ void __launch_bounds__(256) scale_rows_kernel(float* rows, long long n_rows, int pass, double* acc) {
  const long long total = n_rows * kNFeat;
  const double cnt = static_cast<double>(n_rows) * kNCep;
  double m0 = 0.0, m1 = 0.0, m2 = 0.0, i0 = 0.0, i1 = 0.0, i2 = 0.0;
  if (pass >= 1) {
    m0 = acc[0] / cnt; m1 = acc[1] / cnt; m2 = acc[2] / cnt;
  }
  if (pass == 2) {  // std == 0 -> inf -> nan rows, as numpy
    i0 = 1.0 / sqrt(acc[3] / cnt); i1 = 1.0 / sqrt(acc[4] / cnt); i2 = 1.0 / sqrt(acc[5] / cnt);
  }
  double p0 = 0.0, p1 = 0.0, p2 = 0.0;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long j = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; j < total; j += stride) {
    const int col = static_cast<int>(j % kNFeat);
    const int g = col / kNCep;
    const double v = static_cast<double>(rows[j]);
    const double mean = g == 0 ? m0 : g == 1 ? m1 : m2;
    if (pass == 0) {
      p0 += g == 0 ? v : 0.0; p1 += g == 1 ? v : 0.0; p2 += g == 2 ? v : 0.0;
    } else if (pass == 1) {
      const double d = v - mean, dd = d * d;
      p0 += g == 0 ? dd : 0.0; p1 += g == 1 ? dd : 0.0; p2 += g == 2 ? dd : 0.0;
    } else {
      rows[j] = static_cast<float>((v - mean) * (g == 0 ? i0 : g == 1 ? i1 : i2));
    }
  }
  if (pass == 2) return;
  __shared__ double s_part[3][8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  {
    const double w0 = warp_sum(p0), w1 = warp_sum(p1), w2 = warp_sum(p2);
    if (lane == 0) { s_part[0][warp] = w0; s_part[1][warp] = w1; s_part[2][warp] = w2; }
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += s_part[threadIdx.x][w];
    atomicAdd(acc + 3 * pass + threadIdx.x, t);
  }
}

// ---- ingest: 16-bit PCM byte streams -> packed int16 (dataset/sph.py:33-63 big-endian decode,
// dataset/file_processing.py:87-94 STM segment concatenation) --------------------------------------------
// Segment i copies len[i] samples starting at sample index src[i] of the raw stream (byte offset 2 src[i]
// from raw) to dst[dst_off[i] ...]; big_endian swaps the two bytes of every sample (NIST SPHERE pcm).
__global__ void __launch_bounds__(256) ingest_kernel(const uint8_t* raw, int big_endian, const long long* src,
                                                     const long long* dst_off, const long long* len, int16_t* dst) {
  const int seg = blockIdx.y;
  const long long n = len[seg];
  const uint16_t* in = reinterpret_cast<const uint16_t*>(raw) + src[seg];
  int16_t* out = dst + dst_off[seg];
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long k = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; k < n; k += stride) {
    uint16_t v = in[k];
    if (big_endian) v = static_cast<uint16_t>((v << 8) | (v >> 8));
    out[k] = static_cast<int16_t>(v);
  }
}

// ---- bench support ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7FEB352Du; x ^= x >> 15; x *= 0x846CA68Bu; x ^= x >> 16;
  return x;
}
// bit-identical to vad_b200/synth.py:synth_utterance
__global__ void synth_kernel(int16_t* out, long long n_utt, long long utt_samples, long long utt_stride, uint32_t seed,
                             long long first_utt) {
  const long long total = n_utt * utt_samples;
  for (long long g = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; g < total;
       g += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long u = g / utt_samples;
    const uint32_t i = static_cast<uint32_t>(g - u * utt_samples);
    const uint32_t key = mix32(mix32(seed ^ 0x9E3779B9u) + static_cast<uint32_t>(first_utt + u));
    const uint32_t a = mix32(key + i);
    const uint32_t b = mix32(a ^ 0x85EBCA6Bu);
    const int s = static_cast<int>((a & 0xFFFFu) + (a >> 16) + (b & 0xFFFFu) + (b >> 16)) - 131070;
    const uint32_t gh = mix32((key ^ 0x5BD1E995u) + (i >> 11));
    const int gain = (gh & 0x1000u) ? static_cast<int>(1500u + (gh & 0xFFFu)) : static_cast<int>(40u + (gh & 0x7Fu));
    out[u * utt_stride + i] = static_cast<int16_t>((s * gain) >> 16);
  }
}

// FP32 FMA-pipe peak: 16 independent chains per thread. variant 0: register operands;
// variant 1: constant-bank multiplicand (the form the mel / DCT / FFN stages use).
template <int VARIANT>
__global__ void __launch_bounds__(256) fp32_peak_kernel(float* sink, int iters, float m, float a) {
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = static_cast<float>(threadIdx.x + i);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int rep = 0; rep < 8; ++rep) {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        if (VARIANT == 0) acc[i] = fmaf(acc[i], m, a);
        else acc[i] = fmaf(acc[i], c_tab.melw[rep * 16 + i], a);
      }
    }
  }
  float s = 0.0f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += acc[i];
  if (s == 123.456f) sink[0] = s;
}
// variant 2: packed FFMA2 (two fp32 FMAs per lane per instruction), 16 independent chains, register
// multiplicand; variant 3: FFMA2 with an immediate (broadcast) multiplicand -- the butterfly form.
template <int VARIANT>
__global__ void __launch_bounds__(256) fp32x2_peak_kernel(float* sink, int iters, float m, float a) {
  float2 acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = make_float2(static_cast<float>(threadIdx.x + i), static_cast<float>(i));
  const float2 m2 = make_float2(m, m + 1e-7f), a2 = make_float2(a, a);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int rep = 0; rep < 8; ++rep) {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        if (VARIANT == 2) acc[i] = __ffma2_rn(acc[i], m2, a2);
        else acc[i] = __ffma2_rn(acc[i], make_float2(1.0000001f, 1.0000001f), a2);
      }
    }
  }
  float s = 0.0f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += acc[i].x + acc[i].y;
  if (s == 123.456f) sink[0] = s;
}
// variant 4: 8 packed FFMA2 chains interleaved with NS scalar FFMA chains (does scalar work ride along on the
// second FMA sub-pipe while packed work holds the first?).  flop per iteration-rep: 8 * 4 + NS * 2.
template <int NS>
__global__ void __launch_bounds__(256) fp32mix_peak_kernel(float* sink, int iters, float m, float a) {
  float2 acc2[8];
  float acc[NS > 0 ? NS : 1];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc2[i] = make_float2(static_cast<float>(threadIdx.x + i), static_cast<float>(i));
#pragma unroll
  for (int i = 0; i < NS; ++i) acc[i] = static_cast<float>(threadIdx.x - i);
  const float2 a2 = make_float2(a, a);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int rep = 0; rep < 8; ++rep) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        acc2[i] = __ffma2_rn(acc2[i], make_float2(1.0000001f, 1.0000001f), a2);
        if (i < NS) acc[i] = fmaf(acc[i], m, a);
      }
    }
  }
  float s = 0.0f;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += acc2[i].x + acc2[i].y;
#pragma unroll
  for (int i = 0; i < NS; ++i) s += acc[i];
  if (s == 123.456f) sink[0] = s;
}

}  // namespace vadb
