"""Float64 restatement of the opt-in front end and operating point, on top of oracle/ref_math.py.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Pre-emphasis and the analysis window restate
python_speech_features (sigproc.preemphasis, the ``winfunc`` applied to each frame); the threshold
is a softmax threshold on p(voiced).  These are NOT pinned to stored reference output
(python_speech_features is not installed here), like the FFN restatement in ref_math.  With the
defaults (preemph 0, no window, no threshold) every function returns what its ref_math
counterpart returns, bit for bit: it calls it.
"""
import numpy as np

from . import ref_math as rm


def preemphasis(pcm, alpha):
    """python_speech_features sigproc.preemphasis: y[0] = x[0], y[n] = x[n] - alpha x[n-1], float64,
    over the whole signal (last axis; the sample before it is never read).  alpha == 0 returns the input."""
    x = np.asarray(pcm)
    if alpha == 0:
        return x
    x = x.astype(np.float64)
    if x.shape[-1] == 0:
        return x
    y = x.copy()
    y[..., 1:] = x[..., 1:] - alpha * x[..., :-1]
    return y


def get_spec_mag(frames, fft_n=rm.FFT_N, window=None):
    """ref_math.get_spec_mag with ``window`` weights multiplied into samples 0..len(window)-1 of each frame
    (after the same float32 cast)."""
    if window is None:
        return rm.get_spec_mag(frames, fft_n)
    x = np.asarray(frames).astype(np.float32).astype(np.float64)
    w = np.asarray(window, dtype=np.float64)
    x = x.copy()
    x[..., :w.shape[0]] *= w
    spec = np.fft.fft(x, fft_n, axis=-1)[..., : fft_n // 2] / float(fft_n)
    return spec.real ** 2 + spec.imag ** 2


def get_mfcc(frames, filterbank, fft_n=rm.FFT_N, mfcc_n=rm.MFCC_NUM, window=None):
    """ref_math.get_mfcc with the window."""
    return rm.get_mfcc_from_spec(get_spec_mag(frames, fft_n, window), filterbank, mfcc_n)


def mfcc_utterance(pcm, filterbank=None, preemph=0.0, window=None):
    """All frame MFCCs of one utterance: pre-emphasis of the whole utterance, split_into_frames, get_mfcc with
    the window -> [T, 13]."""
    if preemph == 0 and window is None:
        return rm.mfcc_utterance(pcm, filterbank)
    if filterbank is None:
        filterbank = rm.get_mel_filterbanks()
    fr = rm.split_into_frames(preemphasis(pcm, preemph))
    if fr.shape[0] == 0:
        return np.zeros((0, rm.MFCC_NUM))
    return get_mfcc(fr, filterbank, window=window)


def p_voiced(logits):
    """softmax(logits)[..., VOICED] in float64 (NaN rows give NaN)."""
    lg = np.asarray(logits, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        z = lg - lg[..., rm.VOICED:rm.VOICED + 1]
        return 1.0 / np.exp(z).sum(axis=-1)


def decide(logits, threshold=None):
    """threshold None or <= 0: ref_math.decide (argmax == VOICED).  Else speech <=> softmax(logits)[1] >=
    threshold; NaN rows are non-speech."""
    if threshold is None or threshold <= 0:
        return rm.decide(logits)
    logits = np.asarray(logits)
    if logits.shape[0] == 0:
        return np.zeros((0,), dtype=np.uint8)
    with np.errstate(invalid="ignore"):
        return (p_voiced(logits) >= threshold).astype(np.uint8)


def vad_utterance(pcm, w, filterbank=None, mode="analyser", preemph=0.0, window=None, threshold=None):
    """ref_math.vad_utterance with the front end and the threshold."""
    c = mfcc_utterance(pcm, filterbank, preemph, window)
    feats = rm.analyser_features(c) if mode == "analyser" else rm.dataset_features(c)
    logits, _ = rm.ffn_forward(feats, w)
    return c, feats, logits, decide(logits, threshold)
