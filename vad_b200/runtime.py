"""Thin object layer over the C ABI: Handle (device tables + FFN weights), Plan (ragged packed
batch -> segment table), StreamBankHandle.  PyTorch is used only to own device / pinned memory
and to name the CUDA stream; every numeric result comes from libvadb200.so kernels."""
import ctypes as C
import os
import pickle

import numpy as np
import torch

from . import _lib
from ._lib import check

MODE_MFCC, MODE_DATASET, MODE_VAD = 0, 1, 2
PCM_S16, PCM_U8, PCM_S24, PCM_S32, PCM_F32, PCM_F64 = 0, 1, 2, 3, 4, 5
FEAT_ANALYSER, FEAT_DATASET = 0, 1
FFN_KEYS = ("W1", "b1", "W2", "b2", "W3", "b3", "W4", "b4")
FFN_SHAPES = {"W1": (39, 64), "b1": (64,), "W2": (64, 32), "b2": (32,), "W3": (32, 16), "b3": (16,),
              "W4": (16, 3), "b4": (3,)}


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def frames_for_length(n_samples):
    """dataset/file_processing.py:99 framing rule (strict '>')."""
    return int(_lib.load().vadb200_frames_for_length(int(n_samples)))


def outputs_for_length(n_samples):
    return int(_lib.load().vadb200_outputs_for_length(int(n_samples)))


def resampled_length(n_samples, src_rate):
    """Samples at 16 kHz of ``n_samples`` at ``src_rate``: ceil(n up / down), as scipy.signal.resample_poly returns."""
    n = int(_lib.load().vadb200_resampled_length(int(n_samples), int(src_rate)))
    if n < 0:
        raise _lib.VadB200Error(-2 if int(n_samples) >= 0 else -1,
                                "unsupported sample rate %r or negative length" % (src_rate,))
    return n


def glorot_ffn(seed=0):
    """Keras-1 Dense default init (glorot_uniform, zero bias) for the 39-64-32-16-3 FFN of
    learning/ffn_trainer.py:104-116 -- stands in for the trained weights the reference never
    ships.  Same generator as oracle.ref_math.glorot_ffn (kept separate: the product may not
    import the oracle)."""
    rng = np.random.default_rng(seed)
    w = {}
    dims = (39, 64, 32, 16, 3)
    for i in range(4):
        lim = np.sqrt(6.0 / (dims[i] + dims[i + 1]))
        w["W%d" % (i + 1)] = rng.uniform(-lim, lim, size=(dims[i], dims[i + 1])).astype(np.float32)
        w["b%d" % (i + 1)] = np.zeros(dims[i + 1], dtype=np.float32)
    return w


def load_ffn_npz(path):
    """Weight container: .npz with W1[39,64] b1[64] W2[64,32] b2 W3[32,16] b3 W4[16,3] b4
    (Keras layout y = x.W + b); replaces model.load_weights (ffn_trainer.py:159-175)."""
    z = np.load(path)
    return {k: np.asarray(z[k], dtype=np.float32) for k in FFN_KEYS}


TREE_KEYS = ("children_left", "children_right", "feature", "threshold", "value", "classes")


def tree_arrays(tree):
    """The arrays vadb200_set_tree takes, as a dict of TREE_KEYS, from a fitted sklearn DecisionTreeClassifier (found
    by its ``tree_`` / ``classes_``, so sklearn is only needed by a caller that already has one), a path to a pickle of
    one (the reference's ``fname``) or to an ``.npz`` written by ``save_tree_npz``, or such a dict.  ``value`` is
    [n_nodes, n_classes] predict_proba rows: class counts (a tree from sklearn < 1.4) are divided by their row sum, as
    that sklearn's predict_proba did."""
    if isinstance(tree, (str, os.PathLike)):
        if str(tree).endswith(".npz"):
            return load_tree_npz(tree)
        with open(tree, "rb") as f:
            tree = pickle.load(f)
    if hasattr(tree, "tree_") and hasattr(tree, "classes_"):
        if getattr(tree, "n_outputs_", 1) != 1:
            raise ValueError("only single-output trees are supported")
        if getattr(tree, "n_features_in_", 39) != 39:
            raise ValueError("the tree must take the 39 window features")
        t = tree.tree_
        d = dict(children_left=t.children_left, children_right=t.children_right, feature=t.feature,
                 threshold=t.threshold, value=np.asarray(t.value)[:, 0, :], classes=tree.classes_)
    elif all(k in tree for k in TREE_KEYS):
        d = {k: tree[k] for k in TREE_KEYS}
    else:
        raise TypeError("expected a fitted DecisionTreeClassifier, a pickle or .npz path, or a dict of %r" % (TREE_KEYS,))
    classes = np.asarray(d["classes"])
    try:
        cls = classes.astype(np.int64)
    except (TypeError, ValueError):
        raise ValueError("class labels must be the ids 0, 1, 2, got %r" % (classes,))
    if not np.array_equal(cls, classes):
        raise ValueError("class labels must be the ids 0, 1, 2, got %r" % (classes,))
    value = np.array(d["value"], dtype=np.float64).reshape(len(np.asarray(d["children_left"])), cls.size)
    s = value.sum(axis=1)
    counts = (s > 0) & (np.abs(s - 1.0) > 1e-9)
    value[counts] /= s[counts, None]
    out = {k: np.ascontiguousarray(d[k], dtype=np.int64) for k in ("children_left", "children_right", "feature")}
    out.update(threshold=np.ascontiguousarray(d["threshold"], dtype=np.float64), value=np.ascontiguousarray(value),
               classes=np.ascontiguousarray(cls))
    return out


def save_tree_npz(path, tree):
    """Write a tree's arrays (``tree_arrays``) to ``path``: a deployment then runs it without sklearn installed."""
    np.savez(path, **tree_arrays(tree))


def load_tree_npz(path):
    z = np.load(path)
    return {k: z[k] for k in TREE_KEYS}


class Handle(object):
    """One per (process, device): owns the mel / DCT / twiddle tables and the FFN weights."""

    def __init__(self, device=None, ffn_weights=None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("vad_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(
            device.index if isinstance(device, torch.device) else device))
        torch.cuda.init()
        with torch.cuda.device(self.device):
            torch.zeros(1, device=self.device)  # make sure the primary context exists
        self._h = C.c_void_p()
        cfg = _lib.Config()
        self.lib.vadb200_default_config(C.byref(cfg))
        check(self.lib.vadb200_create(C.byref(cfg), self.device.index, C.byref(self._h)))
        self.has_ffn = False
        self.has_tree = False
        self.classifier_version = 0   # changes with the classifier a launch captures (weights, tree, threshold)
        if ffn_weights is not None:
            self.set_ffn_weights(ffn_weights)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.vadb200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self):
        return _stream(self.device)

    def filterbank(self):
        out = np.empty((26, 256), dtype=np.float64)
        check(self.lib.vadb200_get_filterbank(self._h, out.ctypes.data_as(C.c_void_p)))
        return out

    def set_ffn_weights(self, w):
        arrs = []
        for k in FFN_KEYS:
            a = np.ascontiguousarray(np.asarray(w[k], dtype=np.float32))
            if a.shape != FFN_SHAPES[k]:
                raise ValueError("FFN weight %s must have shape %r, got %r" % (k, FFN_SHAPES[k], a.shape))
            arrs.append(a)
        check(self.lib.vadb200_set_ffn_weights(self._h, *[a.ctypes.data_as(C.c_void_p) for a in arrs]))
        self.has_ffn = True
        self.classifier_version += 1

    # ---- decision tree ------------------------------------------------------------------------------
    def set_tree(self, tree):
        """Classify with a decision tree on every VAD path of this handle: a fitted sklearn DecisionTreeClassifier, a
        path to a pickle of one or to an .npz of its arrays (``tree_arrays``).  The decision matches sklearn's
        predict (argmax) or predict_proba[:, 1] >= threshold exactly on the features the device computes; logits
        outputs receive float32 predict_proba by class id.  FFN weights stay set underneath (``clear_tree``)."""
        a = tree_arrays(tree)
        n = int(a["children_left"].shape[0])
        for k in ("children_right", "feature", "threshold"):
            if a[k].shape != (n,):
                raise ValueError("%s must have %d entries" % (k, n))
        p = {k: v.ctypes.data_as(C.c_void_p) for k, v in a.items()}
        check(self.lib.vadb200_set_tree(self._h, n, p["children_left"], p["children_right"], p["feature"],
                                        p["threshold"], p["value"], p["classes"], int(a["classes"].size)))
        self.has_tree = n > 0
        self.classifier_version += 1

    def clear_tree(self):
        """Back to the FFN (if its weights are set)."""
        check(self.lib.vadb200_clear_tree(self._h))
        self.has_tree = False
        self.classifier_version += 1

    @property
    def has_classifier(self):
        return self.has_ffn or self.has_tree

    @property
    def tree_node_count(self):
        return int(self.lib.vadb200_tree_node_count(self._h))

    @property
    def tree_depth(self):
        return int(self.lib.vadb200_tree_depth(self._h))

    def tree_predict(self, x):
        """Feature rows [n, 39] -> (labels uint8 [n], probabilities float32 [n, 3] by class id), CUDA tensors."""
        t = torch.as_tensor(x).to(device=self.device, dtype=torch.float32).contiguous().reshape(-1, 39)
        n = t.shape[0]
        labels = torch.empty((n,), dtype=torch.uint8, device=self.device)
        proba = torch.empty((n, 3), dtype=torch.float32, device=self.device)
        check(self.lib.vadb200_tree_predict(self._h, _ptr(t), n, _ptr(labels), _ptr(proba), self.stream))
        return labels, proba

    def set_ffn_impl(self, impl):
        """0 / "fp32": CUDA-core FFMA; 1 / "tc": tcgen05 kind::tf32 on hi/lo operands; 2 / "tc16" (default):
        tcgen05 kind::f16 on statically scaled fp16 hi/lo operands (half the MMAs; falls back to "tc" for
        weights whose scales would be out of range)."""
        impl = {"fp32": 0, "tc": 1, "tc16": 2}.get(impl, impl)
        check(self.lib.vadb200_set_ffn_impl(self._h, int(impl)))

    @property
    def ffn_impl(self):
        return int(self.lib.vadb200_get_ffn_impl(self._h))

    # ---- opt-in front end and operating point ---------------------------------------------------
    def set_frontend(self, preemph=0.0, window=None):
        """Pre-emphasis y[n] = x[n] - preemph x[n-1] over each utterance (stream, or frame in the per-frame API), then
        a 400-point window: an array of 400 weights or "hamming" (np.hamming(400)); None = rectangular.  The defaults
        are the reference front end."""
        if isinstance(window, str):
            if window != "hamming":
                raise ValueError("window must be an array of 400 weights, 'hamming' or None")
            window = np.hamming(400)
        win = None
        if window is not None:
            win = np.ascontiguousarray(np.asarray(window, dtype=np.float32))
            if win.shape != (400,):
                raise ValueError("window must have 400 weights, got shape %r" % (win.shape,))
        check(self.lib.vadb200_set_frontend(self._h, float(preemph),
                                            win.ctypes.data_as(C.c_void_p) if win is not None else C.c_void_p(0)))

    def frontend(self):
        """(preemph, window as float32[400] or None)."""
        a = C.c_float()
        has = C.c_int()
        win = np.empty(400, dtype=np.float32)
        check(self.lib.vadb200_get_frontend(self._h, C.byref(a), win.ctypes.data_as(C.c_void_p), C.byref(has)))
        return float(a.value), (win if has.value else None)

    def set_decision_threshold(self, p=None):
        """speech <=> softmax(logits)[1] >= p; None (or p <= 0) restores argmax == VOICED."""
        check(self.lib.vadb200_set_decision_threshold(self._h, 0.0 if p is None else float(p)))
        self.classifier_version += 1

    def decision_threshold(self):
        """The threshold on p(voiced), or None for the argmax rule."""
        v = float(self.lib.vadb200_get_decision_threshold(self._h))
        return v if v > 0.0 else None

    # ---- per-frame API --------------------------------------------------------------------
    def _frames_tensor(self, frames):
        t = torch.as_tensor(np.asarray(frames, dtype=np.float32) if not torch.is_tensor(frames) else frames)
        t = t.to(device=self.device, dtype=torch.float32)
        if t.dim() == 1:
            t = t[None]
        return t.contiguous()

    def spec_frames(self, frames):
        t = self._frames_tensor(frames)
        out = torch.empty((t.shape[0], 256), dtype=torch.float32, device=self.device)
        check(self.lib.vadb200_spec_frames(self._h, _ptr(t), t.shape[0], t.shape[1], _ptr(out), self.stream))
        return out

    def mfcc_frames(self, frames):
        t = self._frames_tensor(frames)
        out = torch.empty((t.shape[0], 13), dtype=torch.float32, device=self.device)
        check(self.lib.vadb200_mfcc_frames(self._h, _ptr(t), t.shape[0], t.shape[1], _ptr(out), self.stream))
        return out

    def mfcc_from_spec(self, spec):
        t = self._frames_tensor(spec)
        if t.shape[1] != 256:
            raise ValueError("spectrum must have fft_n/2 = 256 bins")
        out = torch.empty((t.shape[0], 13), dtype=torch.float32, device=self.device)
        check(self.lib.vadb200_mfcc_from_spec(self._h, _ptr(t), t.shape[0], _ptr(out), self.stream))
        return out

    def vad_windows(self, windows, feat_mode=FEAT_ANALYSER, want_feats=False):
        t = torch.as_tensor(windows).to(device=self.device, dtype=torch.float32).contiguous().reshape(-1, 5, 13)
        n = t.shape[0]
        labels = torch.empty((n,), dtype=torch.uint8, device=self.device)
        logits = torch.empty((n, 3), dtype=torch.float32, device=self.device)
        feats = torch.empty((n, 39), dtype=torch.float32, device=self.device) if want_feats else None
        check(self.lib.vadb200_vad_windows(self._h, _ptr(t), n, feat_mode, _ptr(labels), _ptr(logits), _ptr(feats),
                                           self.stream))
        return labels, logits, feats

    def ffn_predict(self, x):
        t = torch.as_tensor(x).to(device=self.device, dtype=torch.float32).contiguous().reshape(-1, 39)
        n = t.shape[0]
        labels = torch.empty((n,), dtype=torch.uint8, device=self.device)
        logits = torch.empty((n, 3), dtype=torch.float32, device=self.device)
        check(self.lib.vadb200_ffn_predict(self._h, _ptr(t), n, _ptr(labels), _ptr(logits), self.stream))
        return labels, logits

    # ---- bench support ----------------------------------------------------------------------
    def synth_pcm(self, n_utt, utt_samples, seed=1234, first_utt=0, utt_stride=None, out=None):
        utt_stride = utt_samples if utt_stride is None else utt_stride
        if out is None:
            out = torch.zeros((n_utt * utt_stride + 8,), dtype=torch.int16, device=self.device)
        check(self.lib.vadb200_synth_pcm(self._h, _ptr(out), n_utt, utt_samples, utt_stride, seed & 0xFFFFFFFF,
                                         first_utt, self.stream))
        return out

    def fp32_peak(self, variant=0, iters=4096):
        v = C.c_double()
        check(self.lib.vadb200_fp32_peak(self._h, variant, iters, C.byref(v)))
        return v.value

    def set_host_chunk_samples(self, samples):
        check(self.lib.vadb200_set_host_chunk_samples(self._h, int(samples)))

    def set_plan_segment_frames(self, frames):
        """Override the segment length of plans created afterwards (0 = automatic)."""
        check(self.lib.vadb200_set_plan_segment_frames(self._h, int(frames)))

    # ---- feature sink / ingest ------------------------------------------------------------------
    def scale_rows(self, rows, want_stats=True):
        """dataset/utils.py:5-32 on a packed [n, 39] float32 CUDA tensor, in place.  Returns the six
        statistics (mean x3, population std x3) as a float64 array when want_stats."""
        if not (torch.is_tensor(rows) and rows.is_cuda and rows.dtype == torch.float32 and rows.is_contiguous()
                and rows.dim() == 2 and rows.shape[1] == 39):
            raise TypeError("rows must be a contiguous [n, 39] float32 CUDA tensor")
        stats = np.zeros(6, dtype=np.float64) if want_stats else None
        check(self.lib.vadb200_scale_rows(self._h, _ptr(rows), rows.shape[0],
                                          stats.ctypes.data_as(C.c_void_p) if want_stats else C.c_void_p(0),
                                          self.stream))
        return stats

    def ingest_pcm(self, raw, src_start, dst_start, lengths, out, big_endian=False):
        """Device decode + gather: ``raw`` uint8 CUDA tensor holding 16-bit samples (2-byte aligned),
        segment i = ``lengths[i]`` samples from sample index ``src_start[i]`` to ``out[dst_start[i]:]``."""
        src = torch.as_tensor(np.asarray(src_start, dtype=np.int64)).to(self.device)
        dst = torch.as_tensor(np.asarray(dst_start, dtype=np.int64)).to(self.device)
        ln_host = np.asarray(lengths, dtype=np.int64)
        ln = torch.as_tensor(ln_host).to(self.device)
        if ln_host.size == 0:
            return out
        check(self.lib.vadb200_ingest_pcm(self._h, _ptr(raw), 1 if big_endian else 0, _ptr(src), _ptr(dst), _ptr(ln),
                                          int(ln_host.size), int(ln_host.max()), _ptr(out), self.stream))
        return out


    def decode_pcm(self, raw, fmt, channels, src_start, dst_start, lengths, out, big_endian=False):
        """Device decode + gather of any VADB200_PCM_* format: ``raw`` uint8 CUDA tensor of interleaved frames of
        ``channels`` samples, segment i = ``lengths[i]`` frames from frame ``src_start[i]`` to the float32 tensor
        ``out[dst_start[i]:]`` in int16 units, the mean of the channels."""
        ln_host = np.asarray(lengths, dtype=np.int64)
        if ln_host.size == 0:
            return out
        src = torch.as_tensor(np.asarray(src_start, dtype=np.int64)).to(self.device)
        dst = torch.as_tensor(np.asarray(dst_start, dtype=np.int64)).to(self.device)
        ln = torch.as_tensor(ln_host).to(self.device)
        check(self.lib.vadb200_decode_pcm(self._h, _ptr(raw), int(fmt), int(channels), 1 if big_endian else 0,
                                          _ptr(src), _ptr(dst), _ptr(ln), int(ln_host.size), int(ln_host.max()),
                                          _ptr(out), self.stream))
        return out


class TreeFitter(object):
    """Fits sklearn 1.9's DecisionTreeClassifier(criterion="gini") on the device (vadb200_tree_fit): the tree is
    sklearn's, bit for bit, at every node where sklearn's choice does not depend on its random feature order; where
    features tie on the best proxy the lowest index wins and the node counts in ``tied_nodes``, so tied_nodes == 0
    means sklearn builds this same tree for every random_state.  Reserves its device memory for ``max_rows`` rows
    (about 1.05 KB each).  Fitting installs no tree: pass the result to ``Handle.set_tree``."""

    def __init__(self, handle, max_rows):
        self.handle = handle
        self.lib = handle.lib
        self.max_rows = int(max_rows)
        self._f = C.c_void_p()
        check(self.lib.vadb200_tree_fitter_create(handle._h, self.max_rows, C.byref(self._f)))

    def close(self):
        if getattr(self, "_f", None) is not None and self._f:
            self.lib.vadb200_tree_fitter_destroy(self._f)
            self._f = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def node_count(self):
        return int(self.lib.vadb200_tree_fit_node_count(self._f))

    def fit(self, x, y, max_depth=None, min_samples_split=2, min_samples_leaf=1, min_impurity_decrease=0.0,
            stream=None):
        """x: [n, 39] float32 CUDA tensor, y: [n] uint8 CUDA tensor of class ids 0 / 1 / 2 (rows with a non-finite
        feature are rejected).  Runs on ``stream`` (a torch.cuda.Stream; the handle's by default) and synchronises it.  Returns the dict of
        ``tree_arrays``' keys plus impurity, n_node_samples and tied_nodes."""
        if not (torch.is_tensor(x) and x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 2
                and x.shape[1] == 39):
            raise TypeError("x must be a contiguous [n, 39] float32 CUDA tensor")
        if not (torch.is_tensor(y) and y.is_cuda and y.dtype == torch.uint8 and y.is_contiguous()
                and y.shape == (x.shape[0],)):
            raise TypeError("y must be a contiguous [n] uint8 CUDA tensor")
        p = _lib.TreeFitParams()
        self.lib.vadb200_default_tree_fit_params(C.byref(p))
        p.max_depth = 0 if max_depth is None else int(max_depth)
        p.min_samples_split = int(min_samples_split)
        p.min_samples_leaf = int(min_samples_leaf)
        p.min_impurity_decrease = float(min_impurity_decrease)
        check(self.lib.vadb200_tree_fit(self._f, _ptr(x), _ptr(y), x.shape[0], C.byref(p),
                                        self.handle.stream if stream is None else C.c_void_p(stream.cuda_stream)))
        return self.result()

    def result(self):
        """The last successful fit (see ``fit``)."""
        m = self.node_count
        out = {k: np.empty(m, np.int64) for k in ("children_left", "children_right", "feature", "n_node_samples")}
        out.update(threshold=np.empty(m), impurity=np.empty(m), value=np.empty((m, 3)), classes=np.empty(3, np.int64))
        nk, tied = C.c_int(), C.c_int64()
        a = lambda k: out[k].ctypes.data_as(C.c_void_p)  # noqa: E731
        check(self.lib.vadb200_tree_fit_result(self._f, a("children_left"), a("children_right"), a("feature"),
                                               a("threshold"), a("value"), a("impurity"), a("n_node_samples"),
                                               a("classes"), C.byref(nk), C.byref(tied)))
        out["value"] = np.ascontiguousarray(out["value"].reshape(-1)[:m * nk.value].reshape(m, nk.value))
        out["classes"] = out["classes"][:nk.value].copy()
        out["tied_nodes"] = int(tied.value)
        return out


class Resampler(object):
    """src_rate -> 16 kHz int16 on the device (scipy.signal.resample_poly's filter, rounded half to even and
    saturated; include/vadb200.h).  Owns the tap table; ``run`` only enqueues work."""

    def __init__(self, handle, src_rate):
        self.handle = handle
        self.lib = handle.lib
        self.src_rate = int(src_rate)
        self._r = C.c_void_p()
        check(self.lib.vadb200_resampler_create(handle._h, self.src_rate, C.byref(self._r)))
        g = int(np.gcd(self.src_rate, 16000))
        self.up, self.down = 16000 // g, self.src_rate // g
        self._ws = None

    def close(self):
        if getattr(self, "_r", None) is not None and self._r:
            self.lib.vadb200_resampler_destroy(self._r)
            self._r = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def output_length(self, n):
        """ceil(n up / down) (vadb200_resampled_length), elementwise for an array."""
        return (np.asarray(n, dtype=np.int64) * self.up + self.down - 1) // self.down

    def output_offsets(self, lengths):
        """The packed 8-aligned output offsets ``run`` uses for these input lengths (n_utt + 1 entries)."""
        m = self.output_length(np.asarray(lengths, dtype=np.int64).reshape(-1))
        offs = np.zeros(m.size + 1, dtype=np.int64)
        offs[1:] = np.cumsum((m + 7) // 8 * 8)
        return offs

    def run(self, d_pcm, offsets, lengths, out=None):
        """``d_pcm``: 1-D int16 (samples) or float32 (int16 units) CUDA tensor; utterance u = lengths[u] samples from
        offsets[u].  Returns (int16 CUDA tensor at 16 kHz, offsets16, lengths16); ``out`` (16-byte aligned int16)
        receives the batch when given."""
        if not (torch.is_tensor(d_pcm) and d_pcm.is_cuda and d_pcm.dim() == 1 and d_pcm.is_contiguous()
                and d_pcm.dtype in (torch.int16, torch.float32)):
            raise TypeError("d_pcm must be a contiguous 1-D int16 or float32 CUDA tensor")
        fmt = PCM_S16 if d_pcm.dtype == torch.int16 else PCM_F32
        offs = np.ascontiguousarray(offsets, dtype=np.int64)
        lens = np.ascontiguousarray(lengths, dtype=np.int64)
        if offs.shape != lens.shape or offs.ndim != 1:
            raise ValueError("offsets and lengths must be 1-D arrays of equal length")
        if lens.size and int((offs + lens).max()) > d_pcm.numel():
            raise ValueError("an utterance ends past the end of d_pcm")
        n = int(lens.size)
        if out is None:
            out = torch.zeros((int(self.output_offsets(lens)[-1]) + 8,), dtype=torch.int16, device=d_pcm.device)
        out_offs = np.zeros(n + 1, dtype=np.int64)                   # filled by the library
        ws_bytes = int(self.lib.vadb200_resample_workspace_bytes(self._r, n))
        if self._ws is None or self._ws.numel() < ws_bytes or self._ws.device != d_pcm.device:
            self._ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=d_pcm.device)
        check(self.lib.vadb200_resample_packed(self._r, fmt, _ptr(d_pcm), offs.ctypes.data_as(C.c_void_p),
                                               lens.ctypes.data_as(C.c_void_p), n, _ptr(out), out.numel(),
                                               out_offs.ctypes.data_as(C.c_void_p), _ptr(self._ws), ws_bytes,
                                               _stream(d_pcm.device)))
        return out, out_offs[:-1].copy(), self.output_length(lens)


class Plan(object):
    """Segment table for one ragged packed batch (offsets / lengths in samples, host side)."""

    def __init__(self, handle, offsets, lengths, mode):
        self.handle = handle
        self.lib = handle.lib
        self.mode = mode
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.lengths = np.ascontiguousarray(lengths, dtype=np.int64)
        if self.offsets.shape != self.lengths.shape or self.offsets.ndim != 1:
            raise ValueError("offsets and lengths must be 1-D arrays of equal length")
        self.n_utt = int(self.offsets.shape[0])
        self._p = C.c_void_p()
        check(self.lib.vadb200_plan_create(handle._h, self.offsets.ctypes.data_as(C.c_void_p),
                                           self.lengths.ctypes.data_as(C.c_void_p), self.n_utt, mode,
                                           C.byref(self._p)))
        self.total_rows = int(self.lib.vadb200_plan_total_rows(self._p))
        self.segment_frames = int(self.lib.vadb200_plan_segment_frames(self._p))
        self.segment_count = int(self.lib.vadb200_plan_segment_count(self._p))
        self.row_offsets = np.empty(self.n_utt + 1, dtype=np.int64)
        check(self.lib.vadb200_plan_row_offsets(self._p, self.row_offsets.ctypes.data_as(C.c_void_p)))

    def close(self):
        if getattr(self, "_p", None) is not None and self._p:
            self.lib.vadb200_plan_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check_pcm(self, pcm):
        if not (torch.is_tensor(pcm) and pcm.dtype == torch.int16 and pcm.is_contiguous() and pcm.dim() == 1):
            raise TypeError("pcm must be a contiguous 1-D torch.int16 tensor")

    def mfcc(self, pcm, out=None):
        """MODE_MFCC -> [rows, 13]; MODE_DATASET -> [rows, 39] (float32, on pcm's device)."""
        self._check_pcm(pcm)
        width = 13 if self.mode == MODE_MFCC else 39
        if out is None:
            out = torch.empty((self.total_rows, width), dtype=torch.float32, device=pcm.device)
        check(self.lib.vadb200_mfcc_packed(self._p, _ptr(pcm), pcm.numel(), _ptr(out), self.handle.stream))
        return out

    def vad(self, pcm, labels=None, want_logits=False, want_feats=False, feat_mode=FEAT_ANALYSER, logits=None):
        self._check_pcm(pcm)
        dev = pcm.device
        if labels is None:
            labels = torch.empty((self.total_rows,), dtype=torch.uint8, device=dev)
        if logits is None and want_logits:
            logits = torch.empty((self.total_rows, 3), dtype=torch.float32, device=dev)
        feats = torch.empty((self.total_rows, 39), dtype=torch.float32, device=dev) if want_feats else None
        check(self.lib.vadb200_vad_packed(self._p, _ptr(pcm), pcm.numel(), _ptr(labels), _ptr(logits), _ptr(feats),
                                          feat_mode, self.handle.stream))
        return labels, logits, feats

    def mfcc_host(self, pcm_host, out_host=None):
        """MODE_MFCC / MODE_DATASET end to end with HOST tensors: chunked H2D, fused kernel, D2H of the rows."""
        if not (torch.is_tensor(pcm_host) and pcm_host.dtype == torch.int16 and not pcm_host.is_cuda):
            raise TypeError("pcm_host must be a CPU torch.int16 tensor")
        width = 13 if self.mode == MODE_MFCC else 39
        if out_host is None:
            out_host = torch.empty((self.total_rows, width), dtype=torch.float32).pin_memory()
        check(self.lib.vadb200_mfcc_host(self._p, _ptr(pcm_host), pcm_host.numel(), _ptr(out_host)))
        return out_host

    def vad_host(self, pcm_host, labels_host=None, logits_host=None, feat_mode=FEAT_ANALYSER):
        """End to end with HOST tensors (pinned for full PCIe speed): H2D, fused kernel, D2H."""
        if not (torch.is_tensor(pcm_host) and pcm_host.dtype == torch.int16 and not pcm_host.is_cuda):
            raise TypeError("pcm_host must be a CPU torch.int16 tensor")
        if labels_host is None:
            labels_host = torch.empty((self.total_rows,), dtype=torch.uint8).pin_memory()
        check(self.lib.vadb200_vad_host(self._p, _ptr(pcm_host), pcm_host.numel(), _ptr(labels_host),
                                        _ptr(logits_host), feat_mode))
        return labels_host, logits_host


    # ---- speech segments (vad_segments.cuh) ------------------------------------------------------
    def speech_segments(self, labels, min_speech_ms=0, min_silence_ms=0, pad_ms=0, want_smoothed=False):
        """Labels [rows] (uint8 CUDA tensor, nonzero = speech) of a MODE_VAD / MODE_DATASET plan -> smoothed labels and
        speech segments.  In order, per utterance: silences shorter than ``min_silence_ms`` between speech are
        filled, speech runs shorter than ``min_speech_ms`` dropped, and the rest padded by ``pad_ms`` on both sides
        (each ceil(ms / 10) rows, at most 1000; 0 = off).  Returns (segments int64 [k, 2] CUDA tensor of
        [start, end) samples within each utterance, segment_offsets and speech_offsets as host int64 [n_utt + 1],
        smoothed uint8 [rows] CUDA tensor or None).  Synchronises once to read the segment count."""
        if not (torch.is_tensor(labels) and labels.is_cuda and labels.dtype == torch.uint8 and labels.is_contiguous()
                and labels.dim() == 1 and labels.numel() == self.total_rows):
            raise TypeError("labels must be a contiguous uint8 CUDA tensor of the plan's %d rows" % self.total_rows)
        rows = [speech_ms_to_rows(v) for v in (min_speech_ms, min_silence_ms, pad_ms)]
        dev = labels.device
        ws_bytes = int(self.lib.vadb200_plan_speech_workspace_bytes(self._p))
        if ws_bytes < 0:
            raise ValueError("speech segments need a MODE_VAD or MODE_DATASET plan")
        ws = getattr(self, "_speech_ws", None)
        if ws is None or ws.numel() < ws_bytes or ws.device != dev:
            ws = self._speech_ws = torch.empty((max(ws_bytes, 16),), dtype=torch.uint8, device=dev)
        max_segs = int(self.lib.vadb200_plan_max_speech_segments(self._p))
        segs = torch.empty((max(max_segs, 1), 2), dtype=torch.int64, device=dev)
        offs = torch.empty((2, self.n_utt + 1), dtype=torch.int64, device=dev)
        smoothed = torch.empty((self.total_rows,), dtype=torch.uint8, device=dev) if want_smoothed else None
        check(self.lib.vadb200_plan_speech_segments(self._p, _ptr(labels), rows[0], rows[1], rows[2], _ptr(smoothed),
                                                    _ptr(segs), _ptr(offs[0]), _ptr(offs[1]), _ptr(ws), ws_bytes,
                                                    self.handle.stream))
        offs_h = offs.cpu().numpy()
        return segs[:int(offs_h[0, -1])], offs_h[0].copy(), offs_h[1].copy(), smoothed

    def gather_speech(self, pcm, segments, segment_offsets, speech_offsets, out=None):
        """Speech audio of every utterance, concatenated in order: an int16 CUDA tensor whose utterance u part is
        out[speech_offsets[u]:speech_offsets[u + 1]].  The arguments after pcm are speech_segments' output."""
        self._check_pcm(pcm)
        dev = pcm.device
        so = torch.as_tensor(np.asarray(segment_offsets, dtype=np.int64)).to(dev)
        sp_h = np.asarray(speech_offsets, dtype=np.int64)
        sp = torch.as_tensor(sp_h).to(dev)
        if so.numel() != self.n_utt + 1 or sp.numel() != self.n_utt + 1:
            raise ValueError("offsets must have n_utt + 1 entries")
        segs = segments if segments.numel() else torch.zeros((1, 2), dtype=torch.int64, device=dev)
        total = int(sp_h[-1])
        if out is None:
            out = torch.empty((total,), dtype=torch.int16, device=dev)
        check(self.lib.vadb200_plan_gather_speech(self._p, _ptr(pcm), pcm.numel(), _ptr(segs.contiguous()), _ptr(so),
                                                  _ptr(sp), _ptr(out), out.numel(), self.handle.stream))
        return out


def speech_ms_to_rows(ms):
    """Duration in ms -> 10 ms rows for the segment parameters: ceil(ms / 10), which must lie in [0, 1000]."""
    ms = float(ms)
    if not ms >= 0.0:
        raise ValueError("durations must be >= 0 ms")
    rows = int(np.ceil(ms / 10.0))
    if rows > 1000:
        raise ValueError("durations must be at most 10000 ms (1000 rows)")
    return rows


class StreamBankHandle(object):
    """A stream bank.  With ``max_feed_samples`` (1 .. 16000) it is a ragged bank: each feed takes any number of
    samples per stream up to that cap (``feed_ragged_ptr``) instead of one 160-sample chunk (``feed_ptr``).  A ragged
    bank at another ``sample_rate`` takes packets at that rate (the cap counted in its samples) and resamples them to
    16 kHz on the device (vadb200_stream_bank_create_ragged_rate)."""

    def __init__(self, handle, n_streams, max_feed_samples=None, sample_rate=16000):
        self.handle = handle
        self.lib = handle.lib
        self.n = int(n_streams)
        self.max_feed = None if max_feed_samples is None else int(max_feed_samples)
        self.sample_rate = int(sample_rate)
        self._b = C.c_void_p()
        if self.max_feed is None:
            if self.sample_rate != 16000:
                raise ValueError("a fixed bank takes 16 kHz chunks: give max_feed_samples for another sample rate")
            check(self.lib.vadb200_stream_bank_create(handle._h, self.n, C.byref(self._b)))
        elif self.sample_rate == 16000:
            check(self.lib.vadb200_stream_bank_create_ragged(handle._h, self.n, self.max_feed, C.byref(self._b)))
        else:
            check(self.lib.vadb200_stream_bank_create_ragged_rate(handle._h, self.n, self.max_feed, self.sample_rate,
                                                                   C.byref(self._b)))

    def close(self):
        if getattr(self, "_b", None) is not None and self._b:
            self.lib.vadb200_stream_bank_destroy(self._b)
            self._b = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        check(self.lib.vadb200_stream_bank_reset(self._b, self.handle.stream))

    def feed_ptr(self, chunks_ptr, labels_ptr, logits_ptr=0, stream=None):
        check(self.lib.vadb200_stream_feed(self._b, C.c_void_p(chunks_ptr), C.c_void_p(labels_ptr),
                                           C.c_void_p(logits_ptr), stream if stream is not None else self.handle.stream))

    def max_rows_per_feed(self):
        """K: the most rows one ragged feed emits per stream (-1 for a fixed bank)."""
        return int(self.lib.vadb200_stream_bank_max_rows_per_feed(self._b))

    def feed_ragged_ptr(self, samples_ptr, offsets_ptr, counts_ptr, labels_ptr, logits_ptr=0, rows_ptr=0,
                        bounds_ptr=0, stream=None):
        """vadb200_stream_feed_ragged: samples int16, offsets int64 [n + 1], counts int32 [n], labels uint8 [n][K],
        logits float32 [n][K][3], rows uint8 [n][K], bounds int64 [n][K] (0: NULL)."""
        check(self.lib.vadb200_stream_feed_ragged(self._b, C.c_void_p(samples_ptr), C.c_void_p(offsets_ptr),
                                                  C.c_void_p(counts_ptr), C.c_void_p(labels_ptr),
                                                  C.c_void_p(logits_ptr), C.c_void_p(rows_ptr),
                                                  C.c_void_p(bounds_ptr),
                                                  stream if stream is not None else self.handle.stream))

    # ---- speech segments (vadb200_stream_bank_set_speech) -------------------------------------------
    def set_speech(self, min_speech_rows, min_silence_rows, pad_rows):
        """Speech on at (S, G, P) rows, each in [0, 1000]; resets every stream.  Returns the delay D in rows."""
        check(self.lib.vadb200_stream_bank_set_speech(self._b, 1, int(min_speech_rows), int(min_silence_rows),
                                                      int(pad_rows), self.handle.stream))
        return self.speech_delay()

    def disable_speech(self):
        check(self.lib.vadb200_stream_bank_set_speech(self._b, 0, 0, 0, 0, self.handle.stream))

    def speech_delay(self):
        """D rows, or -1 when speech is off."""
        return int(self.lib.vadb200_stream_bank_speech_delay(self._b))

    def feed_speech_ptr(self, chunks_ptr, labels_ptr, logits_ptr=0, rows_ptr=0, bounds_ptr=0, stream=None):
        check(self.lib.vadb200_stream_feed_speech(self._b, C.c_void_p(chunks_ptr), C.c_void_p(labels_ptr),
                                                  C.c_void_p(logits_ptr), C.c_void_p(rows_ptr), C.c_void_p(bounds_ptr),
                                                  stream if stream is not None else self.handle.stream))

    def end_streams_ptr(self, end_ptr, tail_rows_ptr=0, tail_bounds_ptr=0, stream=None):
        check(self.lib.vadb200_stream_bank_end_streams(self._b, C.c_void_p(end_ptr), C.c_void_p(tail_rows_ptr),
                                                       C.c_void_p(tail_bounds_ptr),
                                                       stream if stream is not None else self.handle.stream))


_default = {}


def default_handle(device=None):
    """Process-wide handle per device for the function-style drop-in API (mfcc.py functions)."""
    idx = torch.cuda.current_device() if device is None else int(device)
    if idx not in _default:
        _default[idx] = Handle(idx)
    return _default[idx]


def _handle_get_deltas(self, a, b):
    ta = torch.as_tensor(np.asarray(a, dtype=np.float32) if not torch.is_tensor(a) else a).to(
        device=self.device, dtype=torch.float32).contiguous()
    tb = torch.as_tensor(np.asarray(b, dtype=np.float32) if not torch.is_tensor(b) else b).to(
        device=self.device, dtype=torch.float32).contiguous()
    if ta.shape != tb.shape:
        raise ValueError("operands must have equal shapes")
    out = torch.empty_like(ta)
    check(self.lib.vadb200_get_deltas(self._h, _ptr(ta), _ptr(tb), ta.numel(), _ptr(out), self.stream))
    return out


def _handle_lifter(self, cepstra, L=22):
    t = torch.as_tensor(np.asarray(cepstra, dtype=np.float32) if not torch.is_tensor(cepstra) else cepstra).to(
        device=self.device, dtype=torch.float32).contiguous()
    ncoef = int(t.shape[0]) if t.dim() == 1 else int(t.shape[-1])
    out = torch.empty_like(t)
    check(self.lib.vadb200_lifter(self._h, _ptr(t), t.numel() // max(ncoef, 1), ncoef, int(L), _ptr(out), self.stream))
    return out


Handle.get_deltas = _handle_get_deltas
Handle.lifter = _handle_lifter
