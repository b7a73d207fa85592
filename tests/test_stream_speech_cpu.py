"""CPU: speech segments on the stream bank -- the online form of the smoothing.  The oracle's prefix stability at
delay H = (G - 1) + (S - 1) + P (and that H is the least such delay), the kernels' per-stream step and end drain
(vad_segments.cuh seg_step / seg_end, driven on the host by tests/emul/emul_stream_speech.cpp with the kernels'
struct-of-arrays state and lane-strided drain scratch) against oracle/ref_segments.py, and the argument checks that
fail before any device work."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from oracle import ref_segments as rs
from test_gpu_segments import GRID
from test_segments_cpu import markov_labels

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL = os.path.join(ROOT, "tests", "emul")
SO = os.path.join(EMUL, "libvademul_stream.so")
WARM = 7          # chunks before a stream's first label row


def delay(S, G, P):
    return (G - 1 if G > 1 else 0) + (S - 1 if S > 1 else 0) + P


@pytest.fixture(scope="module")
def emul():
    deps = [os.path.join(EMUL, "emul_stream_speech.cpp"), os.path.join(ROOT, "vad_b200", "csrc", "vad_segments.cuh")]
    if not os.path.isfile(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO,
                               os.path.join(EMUL, "emul_stream_speech.cpp")])
    lib = C.CDLL(SO)
    lib.emul_bank_create.restype = C.c_void_p
    lib.emul_bank_create.argtypes = [C.c_int] * 4
    lib.emul_bank_destroy.argtypes = [C.c_void_p]
    lib.emul_bank_delay.argtypes = [C.c_void_p]
    lib.emul_bank_state_words.restype = C.c_longlong
    lib.emul_bank_state_words.argtypes = [C.c_void_p]
    lib.emul_bank_feed.argtypes = [C.c_void_p] + [C.c_void_p] * 4
    lib.emul_bank_end.argtypes = [C.c_void_p] + [C.c_void_p] * 3
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def simulate(lib, S, G, P, dec, ends=None):
    """Feed decisions dec [T][n] to an emulated bank; ends [T][n] ends streams after tick t, and every stream ends
    after the last tick.  Returns per tick labels / rows / bounds [T][n] and the tails {(t, s): (rows, bounds)}."""
    T, n = dec.shape
    b = lib.emul_bank_create(n, S, G, P)
    assert b
    try:
        D = lib.emul_bank_delay(b)
        assert D == delay(S, G, P)
        labs = np.empty((T, n), np.uint8)
        rows = np.empty((T, n), np.uint8)
        bounds = np.empty((T, n), np.int64)
        tails = {}
        ends = np.zeros((T, n), bool) if ends is None else ends.copy()
        if T:
            ends[-1] = True
        for t in range(T):
            d = np.ascontiguousarray(dec[t], np.uint8)
            lib.emul_bank_feed(b, _p(d), _p(labs[t]), _p(rows[t]), _p(bounds[t]))
            if ends[t].any():
                e = ends[t].astype(np.uint8)
                tr = np.full((n, D), 77, np.uint8)          # rows of streams that do not end stay as they were
                tb = np.full((n, D + 1), 77, np.int64)
                lib.emul_bank_end(b, _p(e), _p(tr), _p(tb))
                for s in np.flatnonzero(e):
                    tails[(t, int(s))] = (tr[s], tb[s])
                assert (tr[e == 0] == 77).all() and (tb[e == 0] == 77).all()
        return D, labs, rows, bounds, tails, ends
    finally:
        lib.emul_bank_destroy(b)


def check_stream(S, G, P, D, labs, rows, bounds, tails, ends, s):
    """Every utterance of stream s against the oracle; returns the utterances' label rows."""
    out = []
    t0 = 0
    for t1 in np.flatnonzero(ends[:, s]):
        L, Ro, Bo = labs[t0:t1 + 1, s], rows[t0:t1 + 1, s], bounds[t0:t1 + 1, s]
        assert (L[:WARM] == 255).all() and (L[WARM:] != 255).all()     # a new signal after every end
        lab = L[L != 255]
        R = len(lab)
        got = Ro[Ro != 255]
        assert len(got) == max(0, R - D)
        n_rows = np.cumsum(L != 255)
        assert np.array_equal(n_rows[Ro != 255], np.arange(len(got)) + D + 1)  # row q is final once row q + D is in
        assert (Bo[Ro == 255] == -1).all()
        tr, tb = tails[(int(t1), s)]
        k = min(R, D)
        assert (tr[k:] == 255).all() and (tb[k + 1:] == -1).all()
        smoothed = np.r_[got, tr[:k]].astype(np.uint8)
        b = np.r_[Bo[Bo != -1], tb[:k + 1][tb[:k + 1] != -1]]
        ref = rs.smooth(lab, S, G, P)
        assert np.array_equal(smoothed, ref)
        assert np.array_equal(b.reshape(-1, 2), rs.segments_of(ref))
        out.append(lab)
        t0 = t1 + 1
    return out


def run_and_check(lib, S, G, P, dec, ends=None):
    D, labs, rows, bounds, tails, ends = simulate(lib, S, G, P, dec, ends)
    return [check_stream(S, G, P, D, labs, rows, bounds, tails, ends, s) for s in range(dec.shape[1])]


# ---- the oracle's online form ---------------------------------------------------------------------------------
def test_oracle_prefix_stable_at_delay_h_and_h_is_tight():
    rng = np.random.default_rng(1)
    late = 0
    for _ in range(1500):
        S, G, P = (int(v) for v in rng.integers(0, 12, 3))
        H = delay(S, G, P)
        x = (rng.random(int(rng.integers(1, 100))) < rng.uniform(0.05, 0.95)).astype(np.uint8)
        full = rs.smooth(x, S, G, P)
        for m in range(len(x) + 1):
            pre = rs.smooth(x[:m], S, G, P)
            if m - H > 0:
                assert np.array_equal(pre[:m - H], full[:m - H])
            if H > 0 and 0 <= m - H < m and pre[m - H] != full[m - H]:
                late += 1       # one row earlier is not yet final for this prefix
    assert late > 0
    # and for each step alone, a prefix of m rows whose row m - H is not yet final
    for S, G, P, x, m in [(4, 0, 0, [1, 1, 1, 1], 3), (0, 4, 0, [1, 0, 0, 0, 1], 4), (0, 0, 4, [0, 0, 0, 0, 1], 4)]:
        x = np.array(x, np.uint8)
        H = delay(S, G, P)
        assert rs.smooth(x[:m], S, G, P)[m - H] != rs.smooth(x, S, G, P)[m - H]


# ---- the kernels' step and drain, emulated ---------------------------------------------------------------------
def edge_runs(S, G):
    """Label rows with runs of G - 1, G, S - 1 and S at the start and the end."""
    parts = []
    for k in (G - 1, G, S - 1, S):
        if k > 0:
            parts.append((np.r_[np.ones(3), np.zeros(k), np.ones(k)]).astype(np.uint8))
            parts.append((np.r_[np.zeros(k), np.ones(k), np.zeros(3)]).astype(np.uint8))
    return parts


@pytest.mark.parametrize("S,G,P", GRID)
def test_emulated_bank_equals_oracle(emul, S, G, P):
    rng = np.random.default_rng(S * 1000003 + G * 1009 + P)
    D = delay(S, G, P)
    T = WARM + max(2 * D + 50, 400)     # past the delay: the rings wrap many times
    n = 140                             # two blocks of the end kernel, the second partial
    dec = np.zeros((T, n), np.uint8)
    for s in range(n):
        kind = s % 4
        if kind == 0:
            dec[:, s] = rng.random(T) < rng.uniform(0.05, 0.95)
        elif kind == 1:
            dec[:, s] = markov_labels(rng, T, [3, 12, 50, 400][s % 4 + (s // 4) % 3]) != 0
        else:
            parts = edge_runs(S, G)
            head = parts[int(rng.integers(len(parts)))] if parts else np.zeros(0, np.uint8)
            tail = parts[int(rng.integers(len(parts)))] if parts else np.zeros(0, np.uint8)
            mid = markov_labels(rng, T, 20) != 0
            col = np.r_[np.zeros(WARM), head, mid][:T]
            col[T - len(tail):] = tail[-T:] if len(tail) else col[T:]
            dec[:, s] = col
    run_and_check(emul, S, G, P, dec)


def test_delay_zero_emits_every_row_at_once(emul):
    rng = np.random.default_rng(2)
    dec = (rng.random((60, 5)) < 0.5).astype(np.uint8)
    D, labs, rows, bounds, tails, ends = simulate(emul, 0, 1, 0, dec)
    assert D == 0
    assert np.array_equal(rows, labs)                         # D = 0 and no step on: rows are the labels
    for s in range(5):
        check_stream(0, 1, 0, D, labs, rows, bounds, tails, ends, s)
        assert tails[(59, s)][0].shape == (0,) and tails[(59, s)][1].shape == (1,)


@pytest.mark.parametrize("S,G,P", [(0, 0, 0), (25, 10, 3), (3, 5, 2)])
def test_end_before_rows_during_warmup_and_restart(emul, S, G, P):
    rng = np.random.default_rng(9)
    T, n = 300, 12
    dec = (rng.random((T, n)) < 0.6).astype(np.uint8)
    ends = np.zeros((T, n), bool)
    ends[0, 0] = True              # after one chunk
    ends[6, 1] = True              # after the whole warm-up, before any row
    ends[7, 2] = True              # after exactly one row
    ends[3, 3] = ends[5, 3] = ends[12, 3] = True   # back-to-back ends
    for s in range(4, n):          # end and restart at different ticks, several utterances each
        for t in rng.choice(T - 1, size=int(rng.integers(1, 5)), replace=False):
            ends[t, s] = True
    utts = run_and_check(emul, S, G, P, dec, ends)
    assert [len(u) for u in utts[0][:1]] == [0] and [len(u) for u in utts[1][:1]] == [0]
    assert len(utts[2][0]) == 1
    assert len(utts[3]) == 4


def test_state_size_and_parameter_range(emul):
    # two rings of ceil(999 / 32) words plus meta and last: 264 bytes a stream at the largest parameters
    b = emul.emul_bank_create(3, 1000, 1000, 1000)
    try:
        assert emul.emul_bank_state_words(b) * 4 == 264
    finally:
        emul.emul_bank_destroy(b)
    for bad in [(-1, 0, 0), (0, 1001, 0), (0, 0, 1001)]:
        assert not emul.emul_bank_create(3, *bad)


@settings(max_examples=150, deadline=None)
@given(st.lists(st.lists(st.integers(0, 1), min_size=0, max_size=50), min_size=1, max_size=6),
       st.integers(0, 8), st.integers(0, 8), st.integers(0, 8))
def test_emulated_bank_property(emul, utts, S, G, P):
    """Utterances fed back to back into one stream, each ended: each matches the oracle on its own."""
    sched = []
    for u in utts:
        sched.append(np.r_[np.zeros(WARM, np.uint8), np.array(u, np.uint8)])
    dec = np.concatenate(sched).reshape(-1, 1)
    ends = np.zeros(dec.shape, bool)
    ends[np.cumsum([len(x) for x in sched]) - 1, 0] = True
    got = run_and_check(emul, S, G, P, dec, ends)[0]
    assert [list(g) for g in got] == [list(u) for u in utts]


# ---- argument checks ----------------------------------------------------------------------------------------
def test_cabi_rejects_null_bank_and_keeps_version():
    from vad_b200 import build, _lib
    build.build()
    lib = _lib.load()
    assert lib.vadb200_stream_bank_set_speech(None, 1, 0, 0, 0, None) == -1
    assert lib.vadb200_stream_bank_set_speech(None, 0, 0, 0, 0, None) == -1
    assert lib.vadb200_stream_bank_speech_delay(None) == -1
    assert lib.vadb200_stream_feed_speech(None, None, None, None, None, None, None) == -1
    assert lib.vadb200_stream_bank_end_streams(None, None, None, None, None) == -1
    assert lib.vadb200_version() == 201


class _NoDevice(object):
    """Stands in for the device side: any use of it fails the test."""

    def __getattr__(self, name):
        raise AssertionError("device work before the argument check: " + name)


def _bank_without_device(n=4, delay_rows=-1):
    from vad_b200.analyser import StreamBank
    b = StreamBank.__new__(StreamBank)
    b.n = n
    b.delay = delay_rows
    b.bank = b.handle = b.stream = _NoDevice()
    return b


def test_python_argument_checks_fail_before_device_work():
    b = _bank_without_device()
    for bad in [dict(min_speech_ms=-1), dict(min_silence_ms=10000.5), dict(pad_ms=20000), dict(pad_ms=float("nan"))]:
        with pytest.raises(ValueError):
            b.set_speech(**bad)
    with pytest.raises(RuntimeError):
        b.feed_speech(np.zeros((4, 160), np.int16))
    for ids in ([4], [-1], [0, 1, 9]):
        with pytest.raises(ValueError):
            b.end_streams(ids)
    b = _bank_without_device(delay_rows=3)
    with pytest.raises(ValueError):
        b.feed_speech(np.zeros((3, 160), np.int16))
