"""CPU: speech segments -- the run oracle (oracle/ref_segments.py) on hand-built cases and against a brute-force
windowed restatement, the smoothing kernel's tile functions (vad_segments.cuh, driven on the host by
tests/emul/emul_segments.cpp through the kernel's tile, halo and chunk index math) against the oracle across tile
edges, and the argument checks that need no GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from oracle import ref_segments as rs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL = os.path.join(ROOT, "tests", "emul")
SO = os.path.join(EMUL, "libvademul_seg.so")


@pytest.fixture(scope="module")
def emul():
    deps = [os.path.join(EMUL, "emul_segments.cpp"), os.path.join(ROOT, "vad_b200", "csrc", "vad_segments.cuh")]
    if not os.path.isfile(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO,
                               os.path.join(EMUL, "emul_segments.cpp")])
    lib = C.CDLL(SO)
    lib.emul_speech_smooth.restype = C.c_longlong
    lib.emul_speech_smooth.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p]
    return lib


def windowed(labels, S, G, P):
    """Brute-force restatement: each row from the rows within G - 1 (+ S - 1, + P) of it, per step."""
    x = (np.asarray(labels) != 0).astype(np.uint8)
    n = len(x)
    s1 = x.copy()
    if G > 1:
        for i in range(n):
            if x[i]:
                continue
            left = [j for j in range(max(0, i - G + 1), i) if x[j]]
            right = [j for j in range(i + 1, min(n, i + G)) if x[j]]
            s1[i] = bool(left and right and right[0] - left[-1] - 1 < G)
    s2 = s1.copy()
    if S > 1:
        for i in range(n):
            if not s1[i]:
                continue
            a = i
            while a > 0 and s1[a - 1] and i - a < S:
                a -= 1
            b = i
            while b + 1 < n and s1[b + 1] and b - a + 1 < S:
                b += 1
            s2[i] = (b - a + 1) >= S
    s3 = s2.copy()
    if P > 0:
        for i in range(n):
            s3[i] = s2[max(0, i - P):min(n, i + P + 1)].any()
    return s3


def seg(rows):
    return np.array([(160 * a + 440, 160 * b + 440) for a, b in rows], np.int64).reshape(-1, 2)


# ---- oracle on hand-built cases -----------------------------------------------------------------------------
def test_oracle_trivial_utterances():
    for R in (0, 1, 7):
        s, g = rs.speech_segments(np.zeros(R, np.uint8), 3, 3, 2)
        assert s.shape == (R,) and not s.any() and g.shape == (0, 2)
    s, g = rs.speech_segments(np.ones(1, np.uint8), 0, 0, 5)
    assert list(s) == [1] and np.array_equal(g, seg([(0, 1)]))
    s, g = rs.speech_segments(np.ones(1, np.uint8), 2, 0, 0)    # a one-row utterance cannot keep a 2-row minimum
    assert list(s) == [0] and g.shape == (0, 2)
    s, g = rs.speech_segments(np.ones(9, np.uint8), 5, 5, 5)
    assert s.all() and np.array_equal(g, seg([(0, 9)]))


def test_oracle_alternating_rows_hit_the_segment_bound():
    for R in (1, 2, 9, 10):
        lab = (np.arange(R) % 2 == 0).astype(np.uint8)
        _, g = rs.speech_segments(lab)
        assert g.shape[0] == (R + 1) // 2
        assert np.array_equal(g, seg([(r, r + 1) for r in range(0, R, 2)]))
    _, g = rs.speech_segments((np.arange(10) % 2 == 0).astype(np.uint8), 0, 2)   # gaps of 1 < 2 filled
    assert np.array_equal(g, seg([(0, 9)]))


@pytest.mark.parametrize("k", [2, 3, 7, 1000])
def test_oracle_thresholds_exactly_and_one_either_side(k):
    for gap in (k - 1, k, k + 1):                    # min_silence: gap < k is filled
        lab = np.r_[np.ones(3), np.zeros(gap), np.ones(3)].astype(np.uint8)
        s, g = rs.speech_segments(lab, 0, k, 0)
        assert s.all() == (gap < k)
        assert g.shape[0] == (1 if gap < k else 2)
    for run in (k - 1, k, k + 1):                    # min_speech: run < k is dropped
        lab = np.r_[np.zeros(4), np.ones(run), np.zeros(4)].astype(np.uint8)
        s, g = rs.speech_segments(lab, k, 0, 0)
        assert s.any() == (run >= k)
    for d in (k - 1, k, k + 1):                      # pad: a row within k of speech becomes speech
        lab = np.zeros(2 * k + 5, np.uint8)
        lab[0] = 1
        s = rs.smooth(lab, 0, 0, k)
        assert s[d] == (d <= k)


def test_oracle_edges_and_nonbinary_labels():
    lab = np.array([0, 0, 1, 1, 0, 0, 0, 3, 255, 0], np.uint8)
    s, g = rs.speech_segments(lab)
    assert list(s) == [0, 0, 1, 1, 0, 0, 0, 1, 1, 0]
    assert np.array_equal(g, seg([(2, 4), (7, 9)]))
    # leading / trailing silence is never filled, however short
    lab = np.array([0, 1, 1, 1, 0], np.uint8)
    assert list(rs.smooth(lab, 0, 1000, 0)) == [0, 1, 1, 1, 0]
    # an edge run counts with the length it has
    lab = np.array([1, 1, 0, 0, 0, 1, 1, 1], np.uint8)
    assert list(rs.smooth(lab, 3, 0, 0)) == [0, 0, 0, 0, 0, 1, 1, 1]
    # padding is clipped to the utterance; steps run in order (fill, drop, pad)
    lab = np.array([1, 0, 1, 0, 0, 0, 0, 0, 1, 0], np.uint8)
    assert list(rs.smooth(lab, 3, 2, 1)) == [1, 1, 1, 1, 0, 0, 0, 0, 0, 0]
    # speech offsets: 160 samples per smoothed speech row
    sm, g, so, sp = rs.batch([lab, np.ones(4, np.uint8), np.zeros(0, np.uint8)], 3, 2, 1)
    assert list(so) == [0, 1, 2, 2] and list(sp) == [0, 640, 1280, 1280]
    assert np.array_equal(g[1], [440, 440 + 640])


def test_oracle_speech_audio():
    pcm = np.arange(3000, dtype=np.int16)
    lab = np.array([1, 0, 0, 1, 1] + [0] * 8, np.uint8)
    _, g = rs.speech_segments(lab)
    audio = rs.speech_audio(pcm, g)
    assert np.array_equal(audio, np.r_[pcm[440:600], pcm[920:1240]])
    assert rs.speech_audio(pcm, np.zeros((0, 2), np.int64)).shape == (0,)


@settings(max_examples=300, deadline=None)
@given(st.lists(st.integers(0, 3), min_size=0, max_size=60), st.integers(0, 6), st.integers(0, 6),
       st.integers(0, 6))
def test_oracle_equals_windowed_restatement(lab, S, G, P):
    lab = np.array(lab, np.uint8)
    assert np.array_equal(rs.smooth(lab, S, G, P), windowed(lab, S, G, P))


def test_ms_to_rows():
    from vad_b200 import runtime
    for f in (rs.ms_to_rows, runtime.speech_ms_to_rows):
        assert [f(v) for v in (0, 0.5, 10, 10.01, 19.99, 250, 10000)] == [0, 1, 1, 2, 2, 25, 1000]
        for bad in (-1, 10000.5, 20000, float("nan")):
            with pytest.raises(ValueError):
                f(bad)


# ---- the kernel's tile functions ------------------------------------------------------------------------------
def markov_labels(rng, n, mean_run):
    out = np.empty(n, np.uint8)
    v, i = int(rng.integers(0, 2)), 0
    while i < n:
        r = int(rng.geometric(1.0 / mean_run))
        out[i:i + r] = v * int(rng.integers(1, 256))
        v ^= 1
        i += r
    return out


def emul_smooth(lib, labels, row_off, S, G, P, tile):
    lab = np.ascontiguousarray(labels, np.uint8)
    ro = np.ascontiguousarray(row_off, np.int64)
    out = np.full(len(lab), 7, np.uint8)
    n = lib.emul_speech_smooth(lab.ctypes.data_as(C.c_void_p), ro.ctypes.data_as(C.c_void_p), len(ro) - 1, S, G, P,
                               tile, out.ctypes.data_as(C.c_void_p))
    assert n >= 0
    return out, n


@pytest.mark.parametrize("S,G,P", [(0, 0, 0), (1, 1, 0), (25, 10, 3), (3, 50, 0), (40, 2, 17), (0, 0, 1000),
                                   (1000, 1000, 1000), (7, 1000, 1)])
@pytest.mark.parametrize("tile", [64, 333, 2048])
def test_emulated_tiles_equal_oracle(emul, S, G, P, tile):
    rng = np.random.default_rng(S * 7919 + G * 31 + P + tile)
    lens = [0, 1, tile - 1, tile, tile + 1, 3 * tile + 17, 5000, 2, 0, 12345]
    row_off = np.r_[0, np.cumsum(lens)].astype(np.int64)
    mean = [3, 12, 50, 400]
    labels = np.concatenate([markov_labels(rng, n, mean[i % 4]) for i, n in enumerate(lens)]).astype(np.uint8)
    out, n_starts = emul_smooth(emul, labels, row_off, S, G, P, tile)
    ref, g, so, sp = rs.batch([labels[row_off[u]:row_off[u + 1]] for u in range(len(lens))], S, G, P)
    assert np.array_equal(out, ref)
    assert n_starts == g.shape[0]


def test_emulated_tiles_never_bridge_utterances(emul):
    # speech ... | ... speech: a short gap across an utterance edge is two utterance edges, not a gap
    labels = np.r_[np.ones(50), np.zeros(3), np.zeros(3), np.ones(50)].astype(np.uint8)
    row_off = np.array([0, 53, 106], np.int64)
    out, n = emul_smooth(emul, labels, row_off, 0, 100, 0, 64)
    assert np.array_equal(out, labels) and n == 2
    out, n = emul_smooth(emul, labels, row_off, 0, 0, 10, 16)   # padding stops at the edge too
    ref = np.r_[np.ones(53), np.zeros(3), np.ones(50)].astype(np.uint8)
    ref[50:53] = 1
    ref[53:56] = 1
    assert np.array_equal(out, ref)


def test_window_index_math(emul):
    out = (C.c_longlong * 5)()
    # first tile of an utterance: no row before it
    emul.emul_speech_window(C.c_longlong(100), 64, C.c_longlong(100), C.c_longlong(1000), 10, out)
    assert list(out) == [100, 74, 0, 0, 64]
    # inner tile: H + 1 rows before, H after
    emul.emul_speech_window(C.c_longlong(500), 64, C.c_longlong(100), C.c_longlong(1000), 10, out)
    assert list(out) == [489, 85, 10, 11, 75]
    # clipped at the utterance end
    emul.emul_speech_window(C.c_longlong(990), 10, C.c_longlong(100), C.c_longlong(1000), 10, out)
    assert list(out) == [979, 21, 10, 11, 21]


# ---- C ABI ----------------------------------------------------------------------------------------------------
def test_cabi_rejects_null_plan():
    from vad_b200 import build, _lib
    build.build()
    lib = _lib.load()
    assert lib.vadb200_plan_max_speech_segments(None) == -1
    assert lib.vadb200_plan_speech_workspace_bytes(None) == -1
    assert lib.vadb200_plan_speech_segments(None, None, 0, 0, 0, None, None, None, None, None, 0, None) == -1
    assert lib.vadb200_plan_gather_speech(None, None, 0, None, None, None, None, 0, None) == -1
    assert lib.vadb200_version() == 201
