/* vadb200.h -- C ABI of the B200-native MFCC + FFN voice-activity-detection hot path.
 *
 * The reference (nameofuser1/vad) is pure Python and has no FFI of its own; its boundary is
 * its Python call surface.  Each entry point below names the reference interface it replaces
 * (paths relative to the reference root).  The Python package `vad_b200` binds this library
 * with ctypes and re-exports the reference's function / class names (INTEGRATION.md).
 *
 * Conventions: every function returns 0 on success or a negative VADB200_E_* code and never
 * throws or aborts; vadb200_last_error() gives a thread-local message.  A *_create function that
 * fails leaves *out NULL and retains nothing it allocated.  A handle is bound to
 * one CUDA device.  The library keeps NO per-handle state in device globals: FFN weights travel
 * with every launch as kernel parameters, so different handles (= different classifiers, as one
 * SKLearnAnalyzer owns one classifier, sklearn_analyser.py:21-35) may be driven from different
 * host threads concurrently; one handle's setters (vadb200_set_*) must not race with its own
 * launches.  "d_" pointers are device memory, "h_" pointers host memory; the caller owns every
 * buffer.  `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream);
 * device-pointer calls only enqueue work, never synchronise and can be captured in CUDA graphs.
 * A plan may be in flight on up to 16 streams at once (each launch takes its own work counter).
 */
#ifndef VADB200_H_
#define VADB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VADB200_VERSION 201

#define VADB200_OK 0
#define VADB200_E_INVALID (-1)      /* bad argument (null, negative, misaligned) */
#define VADB200_E_UNSUPPORTED (-2)  /* configuration other than the reference's config.py:20-27 */
#define VADB200_E_CUDA (-3)         /* CUDA runtime error, see vadb200_last_error() */
#define VADB200_E_NOMEM (-4)
#define VADB200_E_STATE (-5)        /* e.g. VAD requested before FFN weights were set */

/* plan modes */
#define VADB200_MODE_MFCC 0     /* rows = all T frames, 13 floats   (mfcc.get_mfcc per frame) */
#define VADB200_MODE_DATASET 1  /* rows = T-5, 39 floats [c,d1,d2]  (file_processing.process_file) */
#define VADB200_MODE_VAD 2      /* rows = T-5, uint8 label          (SKLearnAnalyzer recipe + FFN) */

/* feature recipes inside the VAD kernel */
#define VADB200_FEAT_ANALYSER 0 /* sklearn_analyser.py:52-69,103-107: z-normalised centre frame */
#define VADB200_FEAT_DATASET 1  /* file_processing.py:51-66: raw c, d1, d2 */

typedef struct vadb200_handle vadb200_handle;
typedef struct vadb200_plan vadb200_plan;
typedef struct vadb200_bank vadb200_bank;
typedef struct vadb200_trainer vadb200_trainer;
typedef struct vadb200_tree_fitter vadb200_tree_fitter;

/* config.py:20-27.  Only the reference values are accepted by the fused kernels. */
typedef struct vadb200_config {
  int32_t sample_rate;  /* SAMPLERATE      16000 */
  int32_t frame_size;   /* FRAME_SIZE      400   */
  int32_t frame_step;   /* FRAME_STEP      160   */
  int32_t fft_n;        /* FFT_N           512   */
  int32_t n_filters;    /* FILTERBANKS_NUM 26    */
  int32_t n_mfcc;       /* MFCC_NUM        13    */
  double low_hz;        /* LOW_HZ          300   */
  double high_hz;       /* HIGH_HZ         8000  */
  int32_t lifter_l;     /* mfcc.lifter L   22    */
  int32_t reserved;
} vadb200_config;

const char* vadb200_last_error(void);
int vadb200_version(void);
void vadb200_default_config(vadb200_config* cfg);

/* dataset/file_processing.py:99 -- `while len(data) - offset > frame_size` (strict '>'). */
int64_t vadb200_frames_for_length(int64_t n_samples);
/* dataset/file_processing.py:40-70 -- the 5-slot ring emits T-5 rows, never flushed. */
int64_t vadb200_outputs_for_length(int64_t n_samples);

/* Replaces the per-process setup of dataset_creator.py:16 / SKLearnAnalyzer.__init__
 * (sklearn_analyser.py:21-35): builds the mel filterbank (mfcc.py:39-56), the folded
 * DCT-II x lifter matrix (mfcc.py:76-78,85-90) and FFT twiddles on `device`. */
int vadb200_create(const vadb200_config* cfg, int device, vadb200_handle** out);
int vadb200_destroy(vadb200_handle* h);

/* The dense [26][256] float64 filterbank the handle uses == mfcc.get_mel_filterbanks(). */
int vadb200_get_filterbank(vadb200_handle* h, double* h_out);

/* FFN of learning/ffn_trainer.py:104-116 (Dense 39-64-32-16-3), Keras layout W:(in,out)
 * row-major, y = x.W + b.  Host pointers; replaces model.load_weights. */
int vadb200_set_ffn_weights(vadb200_handle* h, const float* W1, const float* b1, const float* W2,
                            const float* b2, const float* W3, const float* b3, const float* W4,
                            const float* b4);

/* Where the FFN contraction runs: 0 = FP32 CUDA cores (constant-bank FFMA); 1 = tcgen05 tensor cores,
 * kind::tf32 (operands split hi/lo into three products, fp32 accumulation in TMEM); 2 = tcgen05 kind::f16
 * on statically scaled fp16 hi/lo operands (the default; weights whose scales would be out of range keep
 * impl 1, and vadb200_ffn_predict runs any 128-row tile holding a row beyond the feature bounds on impl 1).
 * All three meet the logit tolerance; applies to vadb200_vad_packed / vadb200_vad_host / vadb200_ffn_predict.
 * For any impl, vadb200_ffn_predict on the feature rows the fused VAD path returns reproduces its labels and
 * logits bit for bit. */
int vadb200_set_ffn_impl(vadb200_handle* h, int impl);
int vadb200_get_ffn_impl(vadb200_handle* h);

/* Opt-in front end and operating point (python_speech_features-style front ends); the defaults reproduce the
 * reference (no pre-emphasis, rectangular window, argmax == VOICED).  Handle state read at launch, like ffn_impl.
 * Pre-emphasis y[0] = x[0], y[n] = x[n] - preemph x[n-1] (preemph in [0, 1]) runs over each utterance as a whole
 * before framing (a bank stream: one signal from its last reset; the per-frame API: each frame on its own); then
 * the 400 window weights h_window (NULL = rectangular) multiply frame samples 0..399.  Applies to
 * vadb200_mfcc_packed / _vad_packed / _mfcc_host / _vad_host / _spec_frames / _mfcc_frames / _stream_feed; the
 * per-frame calls reject a window unless frame_len == 400.  get: h_window (nullable) receives the 400 weights
 * (ones without a window). */
int vadb200_set_frontend(vadb200_handle* h, float preemph, const float* h_window /* [400] or NULL */);
int vadb200_get_frontend(vadb200_handle* h, float* preemph, float* h_window /* nullable */, int* has_window);
/* speech <=> softmax(logits)[1] >= p_voiced; p_voiced <= 0 restores argmax == VOICED (default), >= 1 or NaN is
 * rejected.  Logits and features do not depend on it; rows with non-finite features stay label 0.  Applies to
 * vadb200_vad_packed / _vad_host / _vad_windows / _ffn_predict / _stream_feed.  get: 0 = argmax. */
int vadb200_set_decision_threshold(vadb200_handle* h, float p_voiced);
float vadb200_get_decision_threshold(vadb200_handle* h);

/* ---- decision-tree classifier (a fitted sklearn DecisionTreeClassifier, as realtime_analysis/vad.py loads) ------
 * vadb200_set_tree takes exactly the arrays clf.tree_ and clf.classes_ expose: children_left / children_right (-1 at
 * a leaf), feature, threshold (float64), value [n_nodes][n_classes] (float64, tree_.value[:, 0, :]) and classes_
 * (int64 ids, distinct, ascending, each in {0, 1, 2}, config.py:45-47).  Features are the 39 columns of
 * vadb200_vad_windows' feature rows, in that order.  Malformed input (a child index out of range or not greater than
 * its parent's, a node with two parents or none, a node with one child, a feature outside [0, 39), a class outside
 * {0, 1, 2}, a NaN threshold, a negative or non-finite value, more than 2^26 nodes) returns VADB200_E_INVALID and
 * leaves the handle unchanged.  n_nodes == 0 is vadb200_clear_tree.  Host pointers; drains the device like
 * vadb200_set_ffn_weights, so it must not race the handle's own launches.
 * While a tree is set it is the classifier of vadb200_vad_packed / _vad_host / _vad_windows / _stream_feed /
 * _stream_feed_speech / _stream_feed_ragged (the FFN weights stay set underneath it; vadb200_ffn_predict keeps
 * running the FFN).  The decision is sklearn's, exactly, on the features the device computed:
 *   - a node sends x right when x > t32, t32 the largest float32 <= threshold (round toward -inf; >= FLT_MAX: +inf),
 *     which for float32 x is sklearn's float64 test x <= threshold;
 *   - argmax (threshold <= 0): speech <=> classes_[argmax(value[leaf])] == 1, ties to the first maximum as
 *     np.argmax; class 2 (music) is non-speech;
 *   - threshold p > 0 (vadb200_set_decision_threshold): speech <=> p1 >= (double)p, p1 = value[leaf][class 1] in
 *     float64 (predict_proba's column; 0 when the tree lacks class 1).
 * value is taken as predict_proba, as sklearn >= 1.4 stores it (class fractions); a caller holding class counts
 * divides each row by its sum first.  Where a path returns logits (d_logits / h_logits), a tree writes
 * float32(value[leaf]) there in the columns of class ids 0, 1, 2 (0 for a class the tree lacks).  A row with a
 * non-finite feature gets label 0 and NaN in all three columns, as with the FFN. */
#define VADB200_CLASSIFIER_NONE 0
#define VADB200_CLASSIFIER_FFN 1
#define VADB200_CLASSIFIER_TREE 2
int vadb200_set_tree(vadb200_handle* h, int64_t n_nodes, const int64_t* h_children_left,
                     const int64_t* h_children_right, const int64_t* h_feature, const double* h_threshold,
                     const double* h_value, const int64_t* h_classes, int n_classes);
int vadb200_clear_tree(vadb200_handle* h);
int vadb200_get_classifier(const vadb200_handle* h);         /* VADB200_CLASSIFIER_*; -1 for NULL */
int64_t vadb200_tree_node_count(const vadb200_handle* h);    /* 0 without a tree */
int vadb200_tree_depth(const vadb200_handle* h);             /* internal nodes on the longest path; 0 without */
/* The tree over feature rows d_x [n][39] (classifier.predict duck type): d_labels [n] (nullable) gets the decision
 * above, d_proba [n][3] (nullable) the probabilities.  One launch, no allocation, graph-capturable;
 * VADB200_E_STATE without a tree. */
int vadb200_tree_predict(vadb200_handle* h, const float* d_x, int64_t n, uint8_t* d_labels, float* d_proba,
                         void* stream);

/* ---- ragged packed batches (replaces dataset_creator.process_files' Pool.map over files,
 * dataset_creator.py:53-65, and split_into_frames, file_processing.py:80-103) ---------------
 * Utterance u occupies samples [offsets[u], offsets[u] + lengths[u]) of one int16 buffer;
 * offsets must be ascending multiples of 8 samples (16 bytes).  Row ranges per utterance are
 * contiguous in utterance order (vadb200_plan_row_offsets). */
int vadb200_plan_create(vadb200_handle* h, const int64_t* h_offsets, const int64_t* h_lengths,
                        int64_t n_utt, int mode, vadb200_plan** out);
int vadb200_plan_destroy(vadb200_plan* p);
int64_t vadb200_plan_total_rows(const vadb200_plan* p);
int vadb200_plan_row_offsets(const vadb200_plan* p, int64_t* h_out /* n_utt + 1 */);
/* Work decomposition of a plan: utterances are cut into segments of at most
 * vadb200_plan_segment_frames() consecutive frames (chosen from the batch size: >= 16 segments per
 * persistent CTA, at most 2048 frames).  vadb200_set_plan_segment_frames() overrides the choice
 * for plans created afterwards (0 = automatic; else a multiple of 32 in [64, 2048]); results do
 * not depend on it (tests use it to pin the benchmark's one-segment-per-utterance layout). */
int64_t vadb200_plan_segment_frames(const vadb200_plan* p);
int64_t vadb200_plan_segment_count(const vadb200_plan* p);
int vadb200_set_plan_segment_frames(vadb200_handle* h, int frames);

/* mfcc.get_mfcc over every frame (MODE_MFCC: d_out [rows][13]) or process_file's rows
 * (MODE_DATASET: d_out [rows][39]).  d_pcm must be 16-byte aligned; pcm_len = samples. */
int vadb200_mfcc_packed(vadb200_plan* p, const int16_t* d_pcm, int64_t pcm_len, float* d_out,
                        void* stream);

/* Fused MFCC -> 5-frame features -> FFN -> `argmax == VOICED` (sklearn_analyser.py:46-82 with
 * the FFN as classifier).  d_labels [rows] (1 speech / 0 non-speech); d_logits [rows][3] and
 * d_feats [rows][39] are optional (NULL).  Rows with non-finite features (sigma5 == 0) get
 * label 0 and NaN logits. */
int vadb200_vad_packed(vadb200_plan* p, const int16_t* d_pcm, int64_t pcm_len, uint8_t* d_labels,
                       float* d_logits, float* d_feats, int feat_mode, void* stream);

/* End-to-end variant with HOST buffers: chunks the batch, overlaps H2D copies, the fused kernel
 * and D2H of the labels on internal streams; returns when h_labels is complete.  Pinned host
 * memory gives full PCIe bandwidth; pageable memory works but is slower. */
int vadb200_vad_host(vadb200_plan* p, const int16_t* h_pcm, int64_t pcm_len, uint8_t* h_labels,
                     float* h_logits /* nullable */, int feat_mode);
int vadb200_set_host_chunk_samples(vadb200_handle* h, int64_t samples);
/* The same host-buffer pipeline for MODE_MFCC / MODE_DATASET plans: h_out [rows][13 | 39] float32.
 * Replaces the Pool.map(process_file) step of dataset_creator.process_files
 * (dataset_creator.py:61-65) for a packed batch of decoded files. */
int vadb200_mfcc_host(vadb200_plan* p, const int16_t* h_pcm, int64_t pcm_len, float* h_out);

/* ---- speech segments (MODE_VAD / MODE_DATASET plans) -------------------------------------------
 * Frame decisions -> smoothed labels -> speech segments -> speech-only PCM, on the device.  Per utterance, over
 * its rows (nonzero label = speech), in this order: (1) a non-speech run with speech on both sides and shorter than
 * min_silence_rows becomes speech; (2) a speech run shorter than min_speech_rows becomes non-speech (a run cut by
 * the utterance edge counts with the length it has); (3) a row becomes speech when a speech row lies within
 * pad_rows of it.  0 switches a step off (1 too for steps 1 and 2); each parameter in [0, 1000] rows.  Utterances
 * never interact.  A segment is a maximal smoothed speech run [r0, r1) and covers the samples
 * [160 r0 + 440, 160 r1 + 440) of its utterance (row r classifies frame r + 2 and owns its centre hop), so an
 * utterance has at most ceil(R / 2) segments and 160 samples of speech per smoothed speech row.
 * Both calls only enqueue work (no synchronisation, no allocation) and can be captured in CUDA graphs; scratch
 * comes from the caller's workspace, one per stream when a plan runs on several streams at once. */
int64_t vadb200_plan_max_speech_segments(const vadb200_plan* p);      /* sum over utterances of ceil(R_u / 2) */
int64_t vadb200_plan_speech_workspace_bytes(const vadb200_plan* p);
/* d_segments [max][2] int64: start, end samples within the utterance, utterance after utterance;
 * d_segment_offsets [n_utt + 1]: utterance u owns segments [off[u], off[u + 1]); d_speech_offsets (nullable)
 * [n_utt + 1]: utterance u's speech samples start at off[u] of the gathered output.  d_smoothed (nullable) [rows]
 * receives the smoothed 0/1 labels.  Arrays 8-byte aligned, the workspace 16-byte aligned. */
int vadb200_plan_speech_segments(vadb200_plan* p, const uint8_t* d_labels /* [rows] */,
                                 int min_speech_rows, int min_silence_rows, int pad_rows,
                                 uint8_t* d_smoothed /* nullable [rows] */,
                                 int64_t* d_segments /* [max][2] start, end samples within the utterance */,
                                 int64_t* d_segment_offsets /* [n_utt + 1] */,
                                 int64_t* d_speech_offsets /* nullable [n_utt + 1], samples */,
                                 void* d_workspace, int64_t workspace_bytes, void* stream);
/* Speech audio: every utterance's segments concatenated in order, utterance after utterance, into d_out
 * (16-byte aligned, like d_pcm); writes min(d_speech_offsets[n_utt], out_capacity) samples and nothing past
 * out_capacity.  The three arrays are vadb200_plan_speech_segments' output for this plan. */
int vadb200_plan_gather_speech(vadb200_plan* p, const int16_t* d_pcm, int64_t pcm_len,
                               const int64_t* d_segments, const int64_t* d_segment_offsets,
                               const int64_t* d_speech_offsets, int16_t* d_out /* 16-byte aligned */,
                               int64_t out_capacity, void* stream);

/* ---- feature sink and ingest (the steps either side of the path in the offline flow) --------
 * dataset/utils.py:5-32 scale_features on packed dataset rows d_rows [n_rows][39], in place:
 * one scalar mean and one population std per group {mfcc, d1, d2} over all n_rows x 13 values,
 * accumulated in float64.  h_stats (nullable) receives {mean_mfcc, mean_d1, mean_d2, std_mfcc,
 * std_d1, std_d2}; when given, the call synchronises `stream`. */
int vadb200_scale_rows(vadb200_handle* h, float* d_rows, int64_t n_rows, double* h_stats, void* stream);
/* Decode + gather 16-bit PCM on the device: segment i copies d_len[i] samples starting at sample
 * index d_src_start[i] of the raw byte stream d_raw (2-byte aligned; big_endian != 0 swaps bytes:
 * NIST SPHERE, dataset/sph.py:33-63) to d_dst[d_dst_start[i] ...].  With the .stm segment bounds
 * of dataset/stm_parser.py:5-26 as (start, len) this is split_into_frames' concatenation
 * (dataset/file_processing.py:87-94).  max_len = the largest d_len (host copy, sizes the grid). */
int vadb200_ingest_pcm(vadb200_handle* h, const void* d_raw, int big_endian, const int64_t* d_src_start,
                       const int64_t* d_dst_start, const int64_t* d_len, int n_seg, int64_t max_len,
                       int16_t* d_dst, void* stream);

/* ---- audio at other sample rates and formats (DESIGN.md section 5.8) ------------------------------------------
 * Every other entry point reads 16 kHz mono int16.  These calls turn WAV payloads of any common format, channel
 * count and sample rate into that: decode to float32 in int16 units, then resample to 16 kHz int16. */
#define VADB200_PCM_S16 0   /* 16-bit signed: v = s */
#define VADB200_PCM_U8 1    /* 8-bit unsigned: v = (b - 128) * 256 */
#define VADB200_PCM_S24 2   /* 24-bit signed, packed 3 bytes: v = s / 256 */
#define VADB200_PCM_S32 3   /* 32-bit signed: v = s / 65536 */
#define VADB200_PCM_F32 4   /* IEEE float: v = x * 32768, non-finite samples become 0 */
#define VADB200_PCM_F64 5   /* IEEE double: v = x * 32768 rounded to float32, non-finite samples become 0 */

typedef struct vadb200_resampler vadb200_resampler;

/* Decode + gather: segment i turns d_len[i] frames, starting at frame d_src_start[i] of the raw stream d_raw
 * (interleaved frames of `channels` samples in `format`; big_endian != 0 swaps each sample's bytes), into
 * d_dst[d_dst_start[i] ...] as float32 in int16 units, the mean of the channels (summed in channel order in float32,
 * then divided by `channels`).  d_raw is aligned to the sample size (1 for u8 / s24, 2, 4, 8), channels in [1, 32],
 * n_seg <= 65535, max_len = the largest d_len.  Only enqueues work. */
int vadb200_decode_pcm(vadb200_handle* h, const void* d_raw, int format, int channels, int big_endian,
                       const int64_t* d_src_start, const int64_t* d_dst_start, const int64_t* d_len, int n_seg,
                       int64_t max_len, float* d_dst, void* stream);

/* Resampling from src_rate to 16 kHz.  With g = gcd(src_rate, 16000), up = 16000 / g, down = src_rate / g,
 * half = 10 max(up, down) and h = scipy.signal.firwin(2 half + 1, 1 / max(up, down), window=('kaiser', 5.0)) * up,
 * an utterance x[0 .. n) becomes y[m] = sum_k x[k] h[m down + half - k up] for m < ceil(n up / down) (zero padding at
 * both ends: scipy.signal.resample_poly(x, up, down)), computed in float32 from float32 taps, then rounded half to
 * even and saturated to int16.  Accepted: integer rates in [4000, 384000] with max(up, down) <= 1024; 16000 is the
 * identity (one tap of 1); any other rate is VADB200_E_UNSUPPORTED.
 * vadb200_resampled_length: ceil(n up / down), or -1 for an unsupported rate or n < 0.
 * vadb200_resample_taps: the float64 taps h (h_taps nullable, else 2 half + 1 entries); returns their count or -1. */
int64_t vadb200_resampled_length(int64_t n, int src_rate);
int64_t vadb200_resample_taps(int src_rate, double* h_taps);
/* The resampler owns its float32 polyphase tap table on the handle's device; create allocates and synchronises. */
int vadb200_resampler_create(vadb200_handle* h, int src_rate, vadb200_resampler** out);
int vadb200_resampler_destroy(vadb200_resampler* r);
/* Workspace for a call over n_utt utterances (16-byte aligned device memory; one per stream in flight). */
int64_t vadb200_resample_workspace_bytes(const vadb200_resampler* r, int64_t n_utt);
/* A ragged packed batch: utterance u is h_in_lengths[u] samples of d_in from sample h_in_offsets[u] (in_format
 * VADB200_PCM_S16: int16, 2-byte aligned; VADB200_PCM_F32: float32 in int16 units, 4-byte aligned).  Output
 * utterance u goes to d_out (16-byte aligned) from h_out_offsets[u] (filled: n_utt + 1 entries, each a multiple of 8
 * samples, the last the total), whose length is vadb200_resampled_length of the input's; the 8-sample padding
 * between utterances is not written, nor is anything past h_out_offsets[n_utt], which must be <= out_capacity.
 * Only enqueues work: it allocates nothing, never synchronises and can be captured in a CUDA graph (the work list
 * travels in kernel parameters into the workspace). */
int vadb200_resample_packed(vadb200_resampler* r, int in_format, const void* d_in, const int64_t* h_in_offsets,
                            const int64_t* h_in_lengths, int64_t n_utt, int16_t* d_out, int64_t out_capacity,
                            int64_t* h_out_offsets, void* d_workspace, int64_t workspace_bytes, void* stream);

/* ---- per-frame API (mfcc.py:59-78 as the reference calls it: one float frame at a time;
 * batched here over n explicit frames of frame_len <= 512 float32 samples) ------------------ */
int vadb200_spec_frames(vadb200_handle* h, const float* d_frames, int64_t n, int frame_len,
                        float* d_spec /* [n][256] */, void* stream);
int vadb200_mfcc_frames(vadb200_handle* h, const float* d_frames, int64_t n, int frame_len,
                        float* d_mfcc /* [n][13] */, void* stream);
int vadb200_mfcc_from_spec(vadb200_handle* h, const float* d_spec /* [n][256] */, int64_t n,
                           float* d_mfcc /* [n][13] */, void* stream);

/* 5-frame MFCC windows [n][5][13] (rows t-2..t+2) -> features / logits / labels: the classify
 * step of SKLearnAnalyzer.feed_frame (sklearn_analyser.py:52-71) for whole-frame callers. */
int vadb200_vad_windows(vadb200_handle* h, const float* d_windows, int64_t n, int feat_mode,
                        uint8_t* d_labels /* nullable */, float* d_logits /* nullable [n][3] */,
                        float* d_feats /* nullable [n][39] */, void* stream);
/* classifier.predict duck type (sklearn_analyser.py:71): rows [n][39] -> class in {0,1}.  Caller rows have no
 * MFCC-derived bound, so under impl 2 (fp16 operands) each 128-row tile is checked against the bounds its fp16 scales
 * were chosen for (|c or z| <= 1353, |d1| <= 2706, |d2| <= 5416, per feature group); a tile holding any row beyond
 * them runs on the tf32 operands of impl 1 instead, so any finite row gets finite logits within tolerance. */
int vadb200_ffn_predict(vadb200_handle* h, const float* d_x, int64_t n, uint8_t* d_labels,
                        float* d_logits /* nullable [n][3] */, void* stream);

/* mfcc.get_deltas (mfcc.py:81-82): out = a - b over n floats. */
int vadb200_get_deltas(vadb200_handle* h, const float* d_a, const float* d_b, int64_t n,
                       float* d_out, void* stream);
/* mfcc.lifter (mfcc.py:85-93): rows [n_rows][ncoef] times 1 + (L/2) sin(pi k / L); L <= 0 copies. */
int vadb200_lifter(vadb200_handle* h, const float* d_in, int64_t n_rows, int ncoef, int L,
                   float* d_out, void* stream);

/* ---- streaming (SKLearnAnalyzer.feed_frame, sklearn_analyser.py:46-82, for many streams) ---
 * Each stream owns a 320-sample history (two hops; a frame = history + 80 new samples) and a
 * 5-row MFCC ring on the device.  One feed =
 * one 160-sample (10 ms) chunk per stream; labels_out[i] is the decision for the frame fed
 * 3 frames earlier, or 255 while the ring is filling. */
int vadb200_stream_bank_create(vadb200_handle* h, int n_streams, vadb200_bank** out);
int vadb200_stream_bank_destroy(vadb200_bank* b);
int vadb200_stream_bank_reset(vadb200_bank* b, void* stream);
int vadb200_stream_feed(vadb200_bank* b, const int16_t* d_chunks /* [n][160], device-visible */,
                        uint8_t* d_labels /* [n], device-visible */, float* d_logits /* nullable */,
                        void* stream);

/* Speech segments for the bank (the offline smoothing of vadb200_plan_speech_segments, online).  Each stream counts
 * rows from its last reset or end: a feed whose label is not 255 adds row r (chunk r + 7).  With speech on, the feed
 * of chunk r + 7 + D finalises smoothed row r, D = (G > 1 ? G - 1 : 0) + (S > 1 ? S - 1 : 0) + P rows for
 * G = min_silence_rows, S = min_speech_rows, P = pad_rows: rows[i] is its label (0 / 1, or 255 when no row is
 * final this tick) and bounds[i] is 160 r + 440 when row r opens a segment (speech, after non-speech or at r = 0) or
 * closes one (non-speech after speech), else -1; samples count from the stream's last reset or end.  The rows a
 * stream finalises, with the tail of its end, are exactly the offline smoothing of its non-255 labels.
 * All streams share (S, G, P), each in [0, 1000].  set_speech allocates the segment state for these parameters
 * and resets every stream of the bank; enable = 0 frees it and restores the plain bank (also resetting it).  While
 * speech is on, vadb200_stream_feed advances the segment state too (its rows are discarded) and
 * vadb200_stream_bank_reset clears it.  Feeds and ends allocate nothing, never synchronise and can be captured in a
 * CUDA graph; a graph captured before set_speech holds the previous segment state and must be captured again. */
int vadb200_stream_bank_set_speech(vadb200_bank* b, int enable, int min_speech_rows, int min_silence_rows,
                                   int pad_rows, void* stream);
int vadb200_stream_bank_speech_delay(const vadb200_bank* b);   /* D rows, or -1 when speech is off */
/* vadb200_stream_feed plus the segment step; VADB200_E_STATE when speech is off */
int vadb200_stream_feed_speech(vadb200_bank* b, const int16_t* d_chunks /* [n][160], device-visible */,
                               uint8_t* d_labels /* [n], device-visible */, float* d_logits /* nullable */,
                               uint8_t* d_rows /* nullable [n] */, int64_t* d_bounds /* nullable [n] */,
                               void* stream);
/* Streams with d_end[i] != 0 end and start again; the others are untouched.  With speech on, an ended stream's
 * pending rows (at most D) are resolved as if its utterance stopped at its last row R - 1 (a trailing silence is
 * never filled, a trailing speech run counts with the length it has, the pad is clipped): d_tail_rows[i] gets those
 * rows then 255, d_tail_bounds[i] their bounds, then the close of a segment still open (160 R + 440) or -1, then
 * -1.  Rows of streams that do not end are not written.  Then the stream's history, MFCC ring, fed count,
 * front-end previous sample and segment state are zero: its next chunk starts a new signal (255 labels for 7
 * chunks).  With speech off this is a per-stream reset and the tails are not written. */
int vadb200_stream_bank_end_streams(vadb200_bank* b, const uint8_t* d_end /* [n], device-visible */,
                                    uint8_t* d_tail_rows /* nullable [n][D] */,
                                    int64_t* d_tail_bounds /* nullable [n][D + 1] */, void* stream);

/* Ragged bank: each stream takes any number of samples per feed, from 0 up to max_feed_samples in [1, 16000]
 * (1 s), so streams can be fed packets as they arrive (20 ms = 320 samples, 400, 512, ...) and a stream with nothing
 * new sits a feed out.  A stream that has taken N samples since its last reset or end has completed the frames
 * f >= 0 with 160 f + 400 <= N; completing frame f >= 5 emits row f - 5, the fixed bank's row (chunk r + 7 emits row
 * r): it classifies frame f - 3 from the frames f - 5 .. f - 1.  After N samples a stream has emitted the rows of an
 * offline utterance of N + 1 samples (vadb200_outputs_for_length(N + 1)), bit-identical to the fixed bank's and to
 * the fused fp32 path's.  K = ceil(max_feed_samples / 160) rows at most per stream and feed
 * (vadb200_stream_bank_max_rows_per_feed; -1 for NULL or a fixed bank).
 *
 * vadb200_stream_feed_ragged: stream i takes d_samples[d_offsets[i] .. d_offsets[i + 1]) (d_samples 2-byte aligned;
 * both arrays may be pinned host memory: each sample is read once).  d_counts[i] gets the rows it emitted (0 .. K),
 * d_labels[i][0 .. count) their labels (0 / 1) and 255 in the other slots, d_logits[i][j][3] the logits of rows
 * j < count (other slots are not written).  A length below 0 or above max_feed_samples gets d_counts[i] = -1 and
 * all-255 labels and leaves the stream untouched; the offsets live on the device, so this is the kernel's check.
 * With speech on (vadb200_stream_bank_set_speech) each emitted row runs the segment step in row order: d_rows[i][j]
 * is the smoothed row that row j finalises (255: none) and d_bounds[i][j] its bound (or -1), 255 / -1 past count;
 * both may be NULL (the state still advances), and passing either while speech is off is VADB200_E_STATE.  The
 * front end, threshold and speech settings apply as on the fixed bank; vadb200_stream_bank_reset, _set_speech,
 * _speech_delay and _end_streams work with their meaning above (an end discards the samples that have not completed
 * a frame; its tail takes R = the rows the stream has emitted).  vadb200_stream_feed / _feed_speech on a ragged bank,
 * and vadb200_stream_feed_ragged on a fixed one, are VADB200_E_STATE.  A feed is one kernel launch: it allocates
 * nothing, never synchronises and can be captured in a CUDA graph; the lengths are read on the device, so one graph
 * serves any mix of packet sizes. */
int vadb200_stream_bank_create_ragged(vadb200_handle* h, int n_streams, int max_feed_samples, vadb200_bank** out);
int vadb200_stream_bank_max_rows_per_feed(const vadb200_bank* b);
int vadb200_stream_feed_ragged(vadb200_bank* b, const int16_t* d_samples, const int64_t* d_offsets /* [n + 1] */,
                               int32_t* d_counts /* [n] */, uint8_t* d_labels /* [n][K] */,
                               float* d_logits /* nullable [n][K][3] */, uint8_t* d_rows /* nullable [n][K] */,
                               int64_t* d_bounds /* nullable [n][K] */, void* stream);

/* Ragged bank at another source rate (DESIGN.md section 5.9): each stream takes int16 packets at sample_rate r, a
 * rate vadb200_resampler_create accepts (else VADB200_E_UNSUPPORTED), of 0 .. max_feed_samples samples, the cap in
 * [1, r] (else VADB200_E_INVALID; on failure *out is NULL).  With vadb200_resample_packed's up, down, half and
 * filter, a stream that has taken N source samples since its last reset or end has produced the 16 kHz samples m whose
 * newest input lies inside them, (m down + half) div up <= N - 1: M(N) = 0 if N up <= half, else
 * (N up - 1 - half) div down + 1 of them, bit-identical to vadb200_resample_packed's output on the stream's whole
 * signal (the causal prefix of scipy.signal.resample_poly; latency half / up source samples).  Those samples feed the
 * 16 kHz ragged bank above unchanged: after N source samples a stream has emitted the rows of an offline 16 kHz
 * utterance of M(N) + 1 samples.  One feed adds at most cap16 = ceil(max_feed_samples up / down) <= 16000 samples at
 * 16 kHz, so vadb200_stream_bank_max_rows_per_feed returns ceil(cap16 / 160).
 *
 * vadb200_stream_feed_ragged takes source-rate packets (d_samples / d_offsets may be pinned host memory; a packet
 * sample is read once, apart from the few samples two tiles of one stream share).  A length below 0 or above
 * max_feed_samples gets count -1 and all-255 labels and leaves the stream's source-rate and 16 kHz state untouched.
 * Speech bounds are 16 kHz samples, as vadb200_plan_speech_segments gives them.  _end_streams and _reset also zero the
 * source-rate state: the next packet starts a new signal with zeros before it, and an end discards the source samples
 * whose 16 kHz samples are not yet ready.  A feed is three kernel launches and an end two; both allocate nothing,
 * never synchronise and can be captured in a CUDA graph.  sample_rate 16000 creates exactly
 * vadb200_stream_bank_create_ragged's bank.
 * vadb200_stream_bank_sample_rate: r, 16000 for every other bank, -1 for NULL. */
int vadb200_stream_bank_create_ragged_rate(vadb200_handle* h, int n_streams, int max_feed_samples, int sample_rate,
                                           vadb200_bank** out);
int vadb200_stream_bank_sample_rate(const vadb200_bank* b);

/* ---- FFN training (learning/ffn_trainer.py:104-175) ---------------------------------------
 * model.compile(loss='categorical_crossentropy', optimizer='adadelta') + model.train_on_batch for the
 * 39-64-32-16-3 network: forward, backward and the Adadelta update as two hand-written kernels per step,
 * deterministic (per-CTA partial gradients summed in a fixed order).  Keras-1 defaults: lr 1.0, rho 0.95,
 * eps 1e-8.  A trainer starts from the handle's weights if set (else zeros: call _set_weights); rows
 * d_x [n][39] float32 are what the fused kernels emit (MODE_DATASET rows after vadb200_scale_rows),
 * d_y [n] class ids 0 / 1 / 2 (config.py:45-47).  h_loss (nullable) receives the batch loss before the
 * update, as Keras reports it, and makes the call synchronise `stream`. */
int vadb200_trainer_create(vadb200_handle* h, int64_t max_batch, float lr, float rho, float eps,
                           vadb200_trainer** out);
int vadb200_trainer_destroy(vadb200_trainer* t);
int vadb200_trainer_set_weights(vadb200_trainer* t, const float* W1, const float* b1, const float* W2,
                                const float* b2, const float* W3, const float* b3, const float* W4,
                                const float* b4, int reset_optimizer);
int vadb200_trainer_get_weights(vadb200_trainer* t, float* W1, float* b1, float* W2, float* b2, float* W3,
                                float* b3, float* W4, float* b4);
int vadb200_train_on_batch(vadb200_trainer* t, const float* d_x, const uint8_t* d_y, int64_t n,
                           float* h_loss, void* stream);

/* ---- decision-tree fit (learning/decision_classifier_trainer.py: DecisionTreeClassifier(...).fit(X, y)) -----------
 * The tree sklearn 1.9's DecisionTreeClassifier(criterion="gini", splitter="best", max_features=None, max_depth,
 * min_samples_split, min_samples_leaf, min_impurity_decrease) builds on d_x [n][39] float32 and class ids d_y [n] in
 * {0, 1, 2}, array for array and bit for bit, at every node where sklearn's choice does not depend on its random
 * feature order:
 *   - classes = the ids present, ascending; min_samples_split is raised to 2 min_samples_leaf; max_depth <= 0 is
 *     unbounded.  A node is a leaf when depth >= max_depth, n < min_samples_split, n < 2 min_samples_leaf,
 *     impurity <= DBL_EPSILON, it has no candidate, or improvement + DBL_EPSILON < min_impurity_decrease.
 *   - Within a node sorted by feature f, position p is a candidate iff x[p] > x[p-1] + 1e-7f in float32 and both sides
 *     keep min_samples_leaf rows.  Its proxy is -(n_r g_r) - (n_l g_l), g = 1.0 - sum(count^2) / (n n), in float64
 *     without fused multiply-adds; the threshold is double(x[p-1]) / 2.0 + double(x[p]) / 2.0.
 *   - The maximum proxy wins; within a feature the earliest position, across features THE LOWEST FEATURE INDEX.
 *     sklearn takes the first maximum in an order drawn from random_state, which no level-wise builder can reproduce,
 *     so every fit reports tied_nodes, the nodes where a second feature reached the same float64 maximum:
 *     tied_nodes == 0 => sklearn builds this same tree for every random_state.
 *   - Output in sklearn's numbering (depth-first preorder, left child first): children -1, feature -2 and threshold
 *     -2.0 at leaves; value [nodes][n_classes] = count / n_node_samples (tree_.value[:, 0, :] of sklearn >= 1.4), so
 *     the arrays go to vadb200_set_tree as they are.  The tree depends on neither the row order nor the stream.
 * A fitter owns about 1.05 KB of device memory per max_rows row (max_rows <= 2^30 - 8), allocated at create.  A fit
 * reads one small count per tree level, so it synchronises `stream` and cannot be captured in a CUDA graph (like
 * vadb200_train_on_batch with h_loss).  Bad input (a non-finite feature, a class id > 2, n <= 0 or > max_rows, bad
 * params, a NULL pointer) returns VADB200_E_INVALID; a tree of more than 2^26 nodes is VADB200_E_UNSUPPORTED; either
 * leaves the previous result readable.  The fitter is independent of the handle's classifier (fitting installs no
 * tree) and may be destroyed after its handle. */
typedef struct vadb200_tree_fit_params {
  int32_t max_depth;             /* <= 0: unbounded */
  int32_t min_samples_split;     /* >= 2 */
  int32_t min_samples_leaf;      /* >= 1 */
  int32_t reserved;
  double min_impurity_decrease;  /* >= 0, finite */
} vadb200_tree_fit_params;
void vadb200_default_tree_fit_params(vadb200_tree_fit_params* p);       /* sklearn's defaults */
int vadb200_tree_fitter_create(vadb200_handle* h, int64_t max_rows, vadb200_tree_fitter** out);
int vadb200_tree_fitter_destroy(vadb200_tree_fitter* f);
int vadb200_tree_fit(vadb200_tree_fitter* f, const float* d_x /* [n][39] */, const uint8_t* d_y, int64_t n,
                     const vadb200_tree_fit_params* p, void* stream);    /* synchronises stream */
int64_t vadb200_tree_fit_node_count(const vadb200_tree_fitter* f);       /* 0 before the first fit */
/* The last successful fit; every pointer nullable; VADB200_E_STATE before the first fit. */
int vadb200_tree_fit_result(const vadb200_tree_fitter* f, int64_t* h_children_left, int64_t* h_children_right,
                            int64_t* h_feature, double* h_threshold, double* h_value /* [nodes][n_classes] */,
                            double* h_impurity, int64_t* h_n_node_samples, int64_t* h_classes /* [3] */,
                            int* n_classes, int64_t* tied_nodes);

/* ---- bench support -------------------------------------------------------------------------
 * Counter-based integer synthetic PCM, bit-identical to vad_b200/synth.py. */
int vadb200_synth_pcm(vadb200_handle* h, int16_t* d_out, int64_t n_utt, int64_t utt_samples,
                      int64_t utt_stride, uint32_t seed, int64_t first_utt, void* stream);
/* FP32 FMA-pipe microbenchmark: the roofline denominator (MEASURED_PEAKS.json has none).
 * variant 0: FFMA register operands, 1: FFMA constant-bank operand, 2: packed FFMA2 register operands,
 * 3: packed FFMA2 with an immediate multiplicand, 4 / 5 / 6: 8 FFMA2 chains interleaved with 8 / 4 / 0
 * scalar FFMA chains (sub-pipe co-issue probe).  Returns TFLOP/s (2 flop per FMA). */
int vadb200_fp32_peak(vadb200_handle* h, int variant, int iters, double* tflops_out);
/* number of kernel launches issued by this library since load (for bench's gpu_launches) */
int64_t vadb200_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* VADB200_H_ */
