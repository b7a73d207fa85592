"""Speech segments from frame decisions: this project's own definition (the reference has no such function; its
vad.py:52-72 keeps the frames feed_frame returns, and realtime_analysis/simple_analyzer.py smooths decisions with a
hangover).  A plain sequential restatement over runs, kept independent of the kernels' windowed form
(vad_b200/csrc/vad_segments.cuh).

Per utterance, over its rows (nonzero label = speech), in this order:
  1. a maximal non-speech run with speech on both sides, shorter than ``min_silence_rows``, becomes speech;
  2. a maximal speech run shorter than ``min_speech_rows`` becomes non-speech (edge runs count as they are);
  3. a row becomes speech when a speech row lies within ``pad_rows`` of it (clipped to the utterance).
A segment is a maximal smoothed speech run [r0, r1); it covers the samples [160 r0 + 440, 160 r1 + 440) of the
utterance (row r classifies frame r + 2 and owns that frame's centre hop)."""
import numpy as np

HOP = 160
FIRST = 440
MAX_PARAM = 1000


def ms_to_rows(ms):
    """Rows of 10 ms covering ``ms`` milliseconds: ceil(ms / 10)."""
    ms = float(ms)
    if not ms >= 0:
        raise ValueError("durations must be >= 0 ms")
    rows = int(np.ceil(ms / 10.0))
    if rows > MAX_PARAM:
        raise ValueError("durations must be at most 10 s (1000 rows)")
    return rows


def runs(x):
    """Maximal runs of a 0/1 array as a list of (value, start, end)."""
    out = []
    i, n = 0, len(x)
    while i < n:
        j = i
        while j < n and x[j] == x[i]:
            j += 1
        out.append((int(x[i]), i, j))
        i = j
    return out


def smooth(labels, min_speech_rows=0, min_silence_rows=0, pad_rows=0):
    """Smoothed 0/1 labels of one utterance."""
    x = (np.asarray(labels) != 0).astype(np.uint8)
    n = len(x)
    if min_silence_rows > 1:
        for v, a, b in runs(x):
            if v == 0 and a > 0 and b < n and b - a < min_silence_rows:
                x[a:b] = 1
    if min_speech_rows > 1:
        for v, a, b in runs(x):
            if v == 1 and b - a < min_speech_rows:
                x[a:b] = 0
    if pad_rows > 0:
        y = x.copy()
        for v, a, b in runs(x):
            if v == 1:
                y[max(0, a - pad_rows):min(n, b + pad_rows)] = 1
        x = y
    return x


def segments_of(smoothed):
    """int64 [k, 2] sample ranges of the speech runs of smoothed labels."""
    seg = [(HOP * a + FIRST, HOP * b + FIRST) for v, a, b in runs(smoothed) if v == 1]
    return np.array(seg, dtype=np.int64).reshape(-1, 2)


def speech_segments(labels, min_speech_rows=0, min_silence_rows=0, pad_rows=0):
    """(smoothed labels, segments [k, 2] in samples) of one utterance."""
    s = smooth(labels, min_speech_rows, min_silence_rows, pad_rows)
    return s, segments_of(s)


def speech_audio(pcm, segments):
    """Concatenation of the utterance's segment samples, in order."""
    pcm = np.asarray(pcm)
    parts = [pcm[s:e] for s, e in segments]
    return np.concatenate(parts).astype(np.int16) if parts else np.zeros(0, dtype=np.int16)


def batch(labels_per_utt, min_speech_rows=0, min_silence_rows=0, pad_rows=0):
    """Packed form over utterances: (smoothed rows, segments [k, 2], segment offsets, speech offsets)."""
    sm, segs, so, sp = [], [], [0], [0]
    for lab in labels_per_utt:
        s, g = speech_segments(lab, min_speech_rows, min_silence_rows, pad_rows)
        sm.append(s)
        segs.append(g)
        so.append(so[-1] + g.shape[0])
        sp.append(sp[-1] + HOP * int(s.sum()))
    smoothed = np.concatenate(sm).astype(np.uint8) if sm else np.zeros(0, np.uint8)
    return smoothed, np.concatenate(segs).reshape(-1, 2) if segs else np.zeros((0, 2), np.int64), \
        np.array(so, np.int64), np.array(sp, np.int64)
