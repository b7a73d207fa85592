"""Drop-ins for realtime_analysis/: the ``Analyser`` plugin interface (analyser.py:4-15), a
fused-GPU ``FusedAnalyser`` with SKLearnAnalyzer's exact feed_frame contract
(sklearn_analyser.py:15-130), a ``.predict`` duck-typed ``FFNClassifier``
(sklearn_analyser.py:71) and a many-stream ``StreamBank`` for 10 ms hop chunks."""
import abc
import pickle

import numpy as np
import torch

from . import runtime
from .runtime import FEAT_ANALYSER


def _handle_for(weights, handle):
    """One analyser == one classifier (sklearn_analyser.py:21-35): weights given without an explicit
    handle get a PRIVATE handle, so constructing a second object can never replace the classifier of
    an earlier one.  The process-wide default handle serves only the weight-free mfcc.* functions and
    objects that ask for it explicitly."""
    if weights is None:
        return handle or runtime.default_handle()
    w = runtime.load_ffn_npz(weights) if isinstance(weights, str) else weights
    if handle is None:
        return runtime.Handle(ffn_weights=w)
    handle.set_ffn_weights(w)      # explicit handle: the caller owns it and asked for this
    return handle


class Analyser:
    """realtime_analysis/analyser.py:4-15 (the reference's plugin boundary)."""

    def __init__(self):
        pass

    @abc.abstractmethod
    def load_init_inactive_frames(self, frames):
        return

    @abc.abstractmethod
    def feed_frame(self, frame):
        return


class FFNClassifier(object):
    """Object with ``.predict(X[n,39]) -> ndarray[n]`` of classes in {0, 1}
    (1 = VOICED, config.py:46; the FFN's music class 2 maps to 0), evaluated on the GPU."""

    def __init__(self, weights=None, handle=None):
        self.handle = _handle_for(weights, handle)
        if not self.handle.has_ffn:
            raise RuntimeError("FFNClassifier needs FFN weights")

    def predict(self, x):
        labels, _ = self.handle.ffn_predict(np.asarray(x, dtype=np.float32))
        return labels.cpu().numpy().astype(np.int64)

    def predict_logits(self, x):
        return self.handle.ffn_predict(np.asarray(x, dtype=np.float32))[1].cpu().numpy()


class FusedAnalyser(Analyser):
    """SKLearnAnalyzer (sklearn_analyser.py:15-130) on the GPU.

    ``feed_frame(frame)`` takes one whole frame (float / int array of <= 512 samples, vad.py
    feeds 400), returns None for the first five calls, then the raw frame fed three calls
    earlier when it is classified speech, else None.  ``classifier`` may be: None (use the fused
    FFN with ``ffn_weights``), a path to a pickled object with ``.predict`` (as the reference's
    ``fname``), or such an object; an external classifier receives the reference's (1, 39)
    float64 feature row and anything other than class 0 / 1 raises AssertionError
    (sklearn_analyser.py:76-82).  The reference's spectral subtraction is computed and discarded
    there (sklearn_analyser.py:121-123), so it is not reproduced."""

    FRAMES_BUFFER_SIZE = 5
    NOISE_BUFFER_SIZE = 5
    PROCESSING_FRAME_INDEX = 2

    def __init__(self, classifier=None, sample_rate=16000, fft_n=512, mfcc_num=13, low_hz=300, high_hz=8000,
                 fbank_num=26, ffn_weights=None, handle=None):
        Analyser.__init__(self)
        if (sample_rate, int(fft_n), mfcc_num, low_hz, high_hz, fbank_num) != (16000, 512, 13, 300, 8000, 26):
            raise NotImplementedError("vad_b200 kernels are compiled for the reference configuration only")
        self.sample_rate, self.fft_n, self.mfcc_num = sample_rate, int(fft_n), mfcc_num
        self.low_hz, self.high_hz, self.fbank_num = low_hz, high_hz, fbank_num
        if isinstance(classifier, str):
            with open(classifier, "rb") as f:
                classifier = pickle.load(f)
        self.classifier = classifier
        self.handle = _handle_for(ffn_weights if classifier is None else None, handle)
        self.filterbank = self.handle.filterbank()
        if classifier is None:
            if not self.handle.has_ffn:
                raise RuntimeError("FusedAnalyser needs FFN weights or an external classifier")
        self.frames_buffer = []
        self.frames_mfcc_buffer = []  # device tensors [13]
        self.noise_buffer = []
        self.last_logits = None

    def load_init_inactive_frames(self, frames):
        if len(frames) != FusedAnalyser.NOISE_BUFFER_SIZE:
            raise ValueError("Number of inactive frame must be the same as BUFFER SIZE")
        self.noise_buffer = list(self.handle.spec_frames(np.asarray(frames, dtype=np.float32)))

    def _update_frames_buffers(self, frame):
        m = self.handle.mfcc_frames(np.asarray(frame, dtype=np.float32))[0]
        if len(self.frames_buffer) == FusedAnalyser.FRAMES_BUFFER_SIZE:
            self.frames_buffer.pop(0)
            self.frames_mfcc_buffer.pop(0)
        self.frames_buffer.append(frame)
        self.frames_mfcc_buffer.append(m)

    def feed_frame(self, frame):
        if len(self.frames_buffer) < FusedAnalyser.FRAMES_BUFFER_SIZE:
            self._update_frames_buffers(frame)
            return None
        processing_frame = self.frames_buffer[self.PROCESSING_FRAME_INDEX]
        window = torch.stack(self.frames_mfcc_buffer)[None]
        labels, logits, feats = self.handle.vad_windows(window, FEAT_ANALYSER, want_feats=self.classifier is not None)
        if self.classifier is None:
            cls = int(labels[0].item())
            self.last_logits = logits[0]
        else:
            cls = self.classifier.predict(feats.cpu().numpy().astype(np.float64).reshape(1, -1))
        self._update_frames_buffers(frame)
        if cls == 1:
            return processing_frame
        elif cls == 0:
            return None
        else:
            raise AssertionError('Wrong classifier class')


class StreamBank(object):
    """n concurrent 16 kHz streams fed in 160-sample (10 ms) chunks.

    ``feed(chunks[n,160] int16)`` returns uint8[n]: the decision for the frame completed three
    frames earlier (the reference's feed_frame timing), or 255 while a stream's ring is filling.
    Chunk j completes frame j-2 (= 400 samples ending 80 samples into chunk j).  Per-stream state
    (320-sample history, 5-row MFCC ring) lives on the device; chunk input and label output go
    through pinned host buffers.  A tick is captured once into a CUDA graph and replayed: one graph
    launch per tick.  With ``zero_copy`` (default) the graph is the feed kernel alone: it reads the
    chunks from, and writes the labels to, the pinned host buffers directly over PCIe (each chunk
    sample is read once), which removes the two copy nodes and their scheduling gaps from the tick.

    Speech segments (``set_speech``): every stream also runs the offline smoothing of ``Plan.speech_segments``
    online.  A stream's row r is its label from chunk r + 7 (since its last reset or end); ``feed_speech`` returns
    for each stream the smoothed row finalised this tick, r - D (255: none), and a segment bound: 160 (r - D) + 440
    samples when that row opens or closes a segment, else -1.  ``end_streams`` resolves the last D rows of the
    streams it ends and starts them again, leaving the others untouched.

    Ragged bank (``max_feed_samples``, 1 .. 16000): each tick takes any number of samples per stream, up to that cap
    and including none, through ``feed_samples`` / ``feed_samples_speech`` instead of ``feed`` / ``feed_speech``.  A
    stream's rows are those of the fixed bank fed the same signal: completing frame f >= 5 (samples
    [160 f, 160 f + 400)) emits row f - 5, so one tick returns 0 .. K = ceil(max_feed_samples / 160) rows per stream.
    The packets are packed into one pinned buffer with their offsets, and the captured graph reads the lengths on the
    device: one graph serves every packet mix.  ``end_streams`` discards a stream's samples that have not completed a
    frame."""

    NOT_READY = 255
    max_feed = None          # ragged bank: the cap on one stream's samples per tick

    def __init__(self, n_streams, ffn_weights=None, handle=None, use_graph=True, zero_copy=True,
                 max_feed_samples=None):
        self.handle = _handle_for(ffn_weights, handle)
        if not self.handle.has_ffn:
            raise RuntimeError("StreamBank needs FFN weights")
        self.n = int(n_streams)
        if max_feed_samples is not None:
            self.max_feed = int(max_feed_samples)
            if not 1 <= self.max_feed <= 16000:
                raise ValueError("max_feed_samples must lie in [1, 16000]")
        self.bank = runtime.StreamBankHandle(self.handle, self.n, self.max_feed)
        dev = self.handle.device
        if self.max_feed is None:
            self.h_chunks = torch.zeros((self.n, 160), dtype=torch.int16).pin_memory()
            self.h_labels = torch.zeros((self.n,), dtype=torch.uint8).pin_memory()
            self.h_logits = torch.zeros((self.n, 3), dtype=torch.float32).pin_memory()
            self.d_chunks = torch.zeros((self.n, 160), dtype=torch.int16, device=dev)
            self.d_labels = torch.zeros((self.n,), dtype=torch.uint8, device=dev)
            self.d_logits = torch.zeros((self.n, 3), dtype=torch.float32, device=dev)
        else:
            self.k = self.bank.max_rows_per_feed()
            shapes = dict(samples=((self.n * self.max_feed,), torch.int16), offsets=((self.n + 1,), torch.int64),
                          counts=((self.n,), torch.int32), labels=((self.n, self.k), torch.uint8),
                          logits=((self.n, self.k, 3), torch.float32))
            for name, (shape, dtype) in shapes.items():
                setattr(self, "h_" + name, torch.zeros(shape, dtype=dtype).pin_memory())
                setattr(self, "d_" + name, None if zero_copy else torch.zeros(shape, dtype=dtype, device=dev))
        self.stream = torch.cuda.Stream(device=dev)
        self.use_graph = bool(use_graph)
        self.zero_copy = bool(zero_copy)
        self._graphs = {}
        self.delay = -1          # speech delay D in rows; -1: speech off
        self.h_rows = self.h_bounds = self.d_rows = self.d_bounds = None
        self.d_tail_rows = self.d_tail_bounds = None

    def reset(self):
        self.bank.reset()
        torch.cuda.synchronize(self.handle.device)

    def _enqueue_ragged(self, want_logits, speech):
        names = ["samples", "offsets", "counts", "labels"] + (["logits"] if want_logits else []) + \
            (["rows", "bounds"] if speech else [])
        side = "h_" if self.zero_copy else "d_"
        if not self.zero_copy:
            self.d_samples.copy_(self.h_samples, non_blocking=True)
            self.d_offsets.copy_(self.h_offsets, non_blocking=True)
        ptr = {k: getattr(self, side + k).data_ptr() for k in names}
        self.bank.feed_ragged_ptr(ptr["samples"], ptr["offsets"], ptr["counts"], ptr["labels"], ptr.get("logits", 0),
                                  ptr.get("rows", 0), ptr.get("bounds", 0))
        if not self.zero_copy:
            for k in names[2:]:
                getattr(self, "h_" + k).copy_(getattr(self, "d_" + k), non_blocking=True)

    def _enqueue(self, want_logits, speech=False):
        if self.max_feed is not None:
            self._enqueue_ragged(want_logits, speech)
            return
        if self.zero_copy:   # pinned host memory is device-visible under UVA: no copy nodes
            if speech:
                self.bank.feed_speech_ptr(self.h_chunks.data_ptr(), self.h_labels.data_ptr(),
                                          self.h_logits.data_ptr() if want_logits else 0, self.h_rows.data_ptr(),
                                          self.h_bounds.data_ptr())
            else:
                self.bank.feed_ptr(self.h_chunks.data_ptr(), self.h_labels.data_ptr(),
                                   self.h_logits.data_ptr() if want_logits else 0)
            return
        self.d_chunks.copy_(self.h_chunks, non_blocking=True)
        if speech:
            self.bank.feed_speech_ptr(self.d_chunks.data_ptr(), self.d_labels.data_ptr(),
                                      self.d_logits.data_ptr() if want_logits else 0, self.d_rows.data_ptr(),
                                      self.d_bounds.data_ptr())
            self.h_rows.copy_(self.d_rows, non_blocking=True)
            self.h_bounds.copy_(self.d_bounds, non_blocking=True)
        else:
            self.bank.feed_ptr(self.d_chunks.data_ptr(), self.d_labels.data_ptr(),
                               self.d_logits.data_ptr() if want_logits else 0)
        self.h_labels.copy_(self.d_labels, non_blocking=True)
        if want_logits:
            self.h_logits.copy_(self.d_logits, non_blocking=True)

    def _tick(self, want_logits, speech=False):
        """One H2D + kernel + D2H; returns after the labels are on the host."""
        if self.use_graph:
            key = (want_logits, speech)
            g = self._graphs.get(key)
            if g is None:  # capture once (capturing does not execute: no chunk is consumed)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=self.stream):
                    self._enqueue(want_logits, speech)
                self._graphs[key] = g
            g.replay()                                   # one cudaGraphLaunch on the caller's current stream
            torch.cuda.current_stream(self.handle.device).synchronize()
        else:
            with torch.cuda.stream(self.stream):
                self._enqueue(want_logits, speech)
            self.stream.synchronize()

    def _fixed_only(self, what):
        if self.max_feed is not None:
            raise RuntimeError("%s needs a fixed bank: a ragged bank (max_feed_samples) takes feed_samples" % what)

    def feed(self, chunks, want_logits=False):
        """chunks: array-like int16 [n, 160] on the host.  Blocks until labels are on the host."""
        self._fixed_only("feed")
        src = torch.as_tensor(np.asarray(chunks, dtype=np.int16) if not torch.is_tensor(chunks) else chunks)
        if tuple(src.shape) != (self.n, 160):
            raise ValueError("chunks must have shape (%d, 160)" % self.n)
        self.h_chunks.copy_(src)
        self._tick(want_logits)
        if want_logits:
            return self.h_labels.numpy().copy(), self.h_logits.numpy().copy()
        return self.h_labels.numpy().copy()

    def feed_pinned(self):
        """Low-latency tick: the caller has already written ``self.h_chunks`` (pinned); one graph
        launch (H2D + kernel + D2H) is issued and awaited.  Returns a view of ``self.h_labels``."""
        self._fixed_only("feed_pinned")
        self._tick(False)
        return self.h_labels

    # ---- speech segments ----------------------------------------------------------------------------------------
    def set_speech(self, min_speech_ms=0, min_silence_ms=0, pad_ms=0):
        """Turn speech segments on for every stream, with Plan.speech_segments' parameters and ms -> rows rule
        (each ceil(ms / 10) rows, at most 1000).  Resets the bank; returns the delay D in rows."""
        rows = [runtime.speech_ms_to_rows(v) for v in (min_speech_ms, min_silence_ms, pad_ms)]
        dev = self.handle.device
        self._graphs = {}   # captured ticks hold the previous segment state
        d = self.bank.set_speech(*rows)
        if self.h_rows is None:
            shape = (self.n,) if self.max_feed is None else (self.n, self.k)   # ragged: a slot per row
            self.h_rows = torch.zeros(shape, dtype=torch.uint8).pin_memory()
            self.h_bounds = torch.zeros(shape, dtype=torch.int64).pin_memory()
            self.d_rows = torch.zeros(shape, dtype=torch.uint8, device=dev)
            self.d_bounds = torch.zeros(shape, dtype=torch.int64, device=dev)
        self.d_tail_rows = torch.empty((self.n, d), dtype=torch.uint8, device=dev)
        self.d_tail_bounds = torch.empty((self.n, d + 1), dtype=torch.int64, device=dev)
        torch.cuda.synchronize(dev)
        self.delay = d
        return d

    def disable_speech(self):
        """Back to the plain bank (resets it)."""
        self._graphs = {}
        self.bank.disable_speech()
        torch.cuda.synchronize(self.handle.device)
        self.delay = -1
        self.d_tail_rows = self.d_tail_bounds = None

    def feed_speech(self, chunks):
        """feed() plus the segment step: returns (labels uint8 [n], rows uint8 [n], bounds int64 [n]); see the
        class notes.  Needs set_speech."""
        self._fixed_only("feed_speech")
        if self.delay < 0:
            raise RuntimeError("speech is off: call set_speech first")
        src = torch.as_tensor(np.asarray(chunks, dtype=np.int16) if not torch.is_tensor(chunks) else chunks)
        if tuple(src.shape) != (self.n, 160):
            raise ValueError("chunks must have shape (%d, 160)" % self.n)
        self.h_chunks.copy_(src)
        self._tick(False, speech=True)
        return self.h_labels.numpy().copy(), self.h_rows.numpy().copy(), self.h_bounds.numpy().copy()

    # ---- ragged bank ----------------------------------------------------------------------------------------------
    def _pack(self, chunks):
        """Check every packet, then pack them into the pinned samples / offsets buffers."""
        if self.max_feed is None:
            raise RuntimeError("feed_samples needs a ragged bank: create it with max_feed_samples")
        if len(chunks) != self.n:
            raise ValueError("chunks must hold %d arrays, one per stream" % self.n)
        arrs = [np.asarray(c, dtype=np.int16) for c in chunks]
        for a in arrs:
            if a.ndim != 1:
                raise ValueError("each stream's samples must be a 1-D array")
            if a.shape[0] > self.max_feed:
                raise ValueError("a stream took %d samples, more than max_feed_samples = %d"
                                 % (a.shape[0], self.max_feed))
        flat, off = self.h_samples.numpy(), self.h_offsets.numpy()
        pos = 0
        for i, a in enumerate(arrs):
            off[i] = pos
            flat[pos:pos + a.shape[0]] = a
            pos += a.shape[0]
        off[self.n] = pos

    def _rows_of(self, buf):
        counts = self.h_counts.numpy()
        return [buf[i, :counts[i]].copy() for i in range(self.n)]

    def feed_samples(self, chunks, want_logits=False):
        """chunks: n 1-D int16 arrays, stream i's new samples (0 .. max_feed_samples of them).  Returns n uint8 arrays
        of the rows each stream completed this tick (and n float32 [k, 3] logit arrays).  Blocks until they are on the
        host."""
        self._pack(chunks)
        self._tick(want_logits)
        labels = self._rows_of(self.h_labels.numpy())
        if want_logits:
            return labels, self._rows_of(self.h_logits.numpy())
        return labels

    def feed_samples_speech(self, chunks):
        """feed_samples plus the segment step: for each stream (labels, rows, bounds), aligned with its labels: rows[j]
        is the smoothed row that label j finalises (255: none) and bounds[j] its bound (-1: none).  Needs
        set_speech."""
        if self.max_feed is not None and self.delay < 0:
            raise RuntimeError("speech is off: call set_speech first")
        self._pack(chunks)
        self._tick(False, speech=True)
        return list(zip(self._rows_of(self.h_labels.numpy()), self._rows_of(self.h_rows.numpy()),
                        self._rows_of(self.h_bounds.numpy())))

    def end_streams(self, ids):
        """End the streams ``ids`` and start them again (their next chunk begins a new signal).  With speech on,
        returns for each id (tail_rows uint8 [k], tail_bounds int64 [k + 1]): its k <= D pending smoothed rows, their
        bounds, then the close of a segment still open (160 R + 440 after R rows) or -1.  With speech off the streams
        are reset and each tail is empty."""
        ids = [int(i) for i in np.asarray(ids, dtype=np.int64).reshape(-1)]
        if any(i < 0 or i >= self.n for i in ids):
            raise ValueError("stream ids must lie in [0, %d)" % self.n)
        dev = self.handle.device
        end = np.zeros(self.n, np.uint8)
        end[ids] = 1
        speech = self.delay >= 0
        with torch.cuda.stream(self.stream):
            d_end = torch.as_tensor(end).to(dev, non_blocking=False)
            self.bank.end_streams_ptr(d_end.data_ptr(), self.d_tail_rows.data_ptr() if speech else 0,
                                      self.d_tail_bounds.data_ptr() if speech else 0, stream=self.stream.cuda_stream)
            if speech:
                sel = torch.as_tensor(np.asarray(ids, np.int64)).to(dev)
                rows = self.d_tail_rows.index_select(0, sel).cpu().numpy()
                bounds = self.d_tail_bounds.index_select(0, sel).cpu().numpy()
        self.stream.synchronize()
        if not speech:
            return [(np.zeros(0, np.uint8), np.zeros(0, np.int64)) for _ in ids]
        out = []
        for r, b in zip(rows, bounds):
            k = int(np.count_nonzero(r != 255))
            out.append((r[:k].copy(), b[:k + 1].copy()))
        return out
