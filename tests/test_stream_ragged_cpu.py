"""CPU: the ragged stream bank.  Its sample-ring index math (vad_b200/csrc/vad_ragged.h, driven on the host by
tests/emul/emul_stream_ragged.cpp as stream_ragged_kernel uses it) stages every frame from exactly the signal's
samples and emits the fixed bank's rows for any chunking; the C ABI and the Python surface reject bad arguments
before any device work."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import ref_math as rm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL = os.path.join(ROOT, "tests", "emul")
SO = os.path.join(EMUL, "libvademul_ragged.so")
SIZES = (0, 1, 79, 80, 81, 159, 160, 161, 399, 400, 401)


@pytest.fixture(scope="module")
def emul():
    deps = [os.path.join(EMUL, "emul_stream_ragged.cpp"), os.path.join(ROOT, "vad_b200", "csrc", "vad_ragged.h")]
    if not os.path.isfile(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", SO,
                               os.path.join(EMUL, "emul_stream_ragged.cpp")])
    lib = C.CDLL(SO)
    lib.emul_ragged_stream.restype = C.c_longlong
    lib.emul_ragged_stream.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong] + [C.c_void_p] * 5
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def run(lib, cap, sizes, signal):
    sizes = np.ascontiguousarray(sizes, np.int32)
    signal = np.ascontiguousarray(signal, np.int16)
    m = len(signal) // 160 + 2
    frame = np.full(m, -9, np.int64)
    staged = np.zeros((m, 401), np.int16)
    row = np.full(m, -9, np.int64)
    slot = np.full(m, -9, np.int32)
    counts = np.full(len(sizes), -9, np.int32)
    k = lib.emul_ragged_stream(cap, len(sizes), _p(sizes), _p(signal), m, _p(frame), _p(staged), _p(row), _p(slot),
                               _p(counts))
    assert k >= 0
    return frame[:k], staged[:k], row[:k], slot[:k], counts


def check(lib, cap, sizes, rng):
    sizes = np.asarray(sizes, np.int64)
    n = int(sizes.sum())
    signal = rng.integers(-32768, 32768, n).astype(np.int16)
    frame, staged, row, slot, counts = run(lib, cap, sizes, signal)
    F = rm.n_frames(n + 1)                       # frames with 160 f + 400 <= n
    assert np.array_equal(frame, np.arange(F))
    padded = np.r_[np.zeros(1, np.int16), signal]
    for f in range(F):
        assert np.array_equal(staged[f], padded[160 * f:160 * f + 401]), f
    assert np.array_equal(row, np.where(frame >= 5, frame - 5, -1))
    K = (cap + 159) // 160
    assert lib.emul_ragged_max_rows(cap) == K
    assert counts.max(initial=0) <= K and counts.min(initial=0) >= 0
    N = np.cumsum(sizes)
    assert np.array_equal(np.cumsum(counts), [rm.n_outputs(int(x) + 1) for x in N])
    # a feed's rows take its output slots 0 .. count - 1 in row order
    fed_by = np.searchsorted(N, 160 * frame + 400, side="left")
    for t in np.unique(fed_by[row >= 0]):
        sel = (fed_by == t) & (row >= 0)
        assert np.array_equal(slot[sel], np.arange(counts[t]))
    return F


@pytest.mark.parametrize("cap", [1, 80, 160, 161, 320, 400, 401, 480, 1024, 1600, 16000])
def test_staged_frames_equal_the_signal(emul, cap):
    rng = np.random.default_rng(cap)
    R = emul.emul_ragged_ring_samples(cap)
    assert R % 160 == 0 and R >= cap + 401
    pool = np.array([s for s in SIZES if s <= cap] + [cap])
    frames = 0
    target = max(30 * cap, 8000)
    for trial in range(4):
        if trial == 0:
            sizes = np.full(max(1, target // max(cap, 1)), cap)            # always full
        elif trial == 1:
            sizes = rng.choice(pool, size=max(1, 2 * target // (int(pool.mean()) + 1)))
        elif trial == 2:
            sizes = rng.integers(0, cap + 1, size=max(1, 2 * target // (cap + 1)))
        else:                                                           # bursts between idle stretches
            sizes = np.where(rng.random(max(1, 2 * target // (cap + 1))) < 0.3, cap, 0)
        frames += check(emul, cap, sizes, rng)
    assert frames > 0


def test_zero_and_single_sample_feeds(emul):
    rng = np.random.default_rng(3)
    sizes = np.r_[np.zeros(5, np.int64), np.ones(1200, np.int64), np.zeros(3, np.int64), [401, 0, 399]]
    assert check(emul, 401, sizes, rng) == rm.n_frames(int(sizes.sum()) + 1)


def test_bad_sizes_are_refused(emul):
    for sizes in ([161], [-1], [0, 200, 0]):
        sig = np.zeros(400, np.int16)
        s = np.asarray(sizes, np.int32)
        m = 8
        out = [np.zeros(m, np.int64), np.zeros((m, 401), np.int16), np.zeros(m, np.int64), np.zeros(m, np.int32),
               np.zeros(len(s), np.int32)]
        assert emul.emul_ragged_stream(160, len(s), _p(s), _p(sig), m, *[_p(a) for a in out]) == -1


# ---- argument checks ----------------------------------------------------------------------------------------
def test_cabi_rejects_bad_arguments_and_keeps_version():
    from vad_b200 import build, _lib
    build.build()
    lib = _lib.load()
    out = C.c_void_p(12345)
    assert lib.vadb200_stream_bank_create_ragged(None, 4, 160, C.byref(out)) == -1
    assert not out.value                                  # a failed create leaves *out NULL
    fake = C.create_string_buffer(64)                     # never dereferenced: the cap check comes first
    for cap in (0, 16001, -5):
        out = C.c_void_p(12345)
        assert lib.vadb200_stream_bank_create_ragged(C.cast(fake, C.c_void_p), 4, cap, C.byref(out)) == -1
        assert not out.value
    assert lib.vadb200_stream_bank_create_ragged(C.cast(fake, C.c_void_p), 0, 160, C.byref(out)) == -1
    assert lib.vadb200_stream_bank_create_ragged(C.cast(fake, C.c_void_p), 4, 160, None) == -1
    assert lib.vadb200_stream_bank_max_rows_per_feed(None) == -1
    assert lib.vadb200_stream_feed_ragged(None, None, None, None, None, None, None, None, None) == -1
    assert lib.vadb200_version() == 201


class _NoDevice(object):
    """Stands in for the device side: any use of it fails the test."""

    def __getattr__(self, name):
        raise AssertionError("device work before the argument check: " + name)


def _bank_without_device(n=4, cap=None, delay_rows=-1):
    from vad_b200.analyser import StreamBank
    b = StreamBank.__new__(StreamBank)
    b.n = n
    b.delay = delay_rows
    if cap is not None:
        b.max_feed = cap
        b.k = (cap + 159) // 160
    b.bank = b.handle = b.stream = _NoDevice()
    b.h_samples = b.h_offsets = _NoDevice()
    return b


def test_python_argument_checks_fail_before_device_work():
    from vad_b200.analyser import StreamBank
    with pytest.raises(ValueError):
        StreamBank.__init__(_bank_without_device(), 4, handle=_Weighted(), max_feed_samples=16001)
    with pytest.raises(ValueError):
        StreamBank.__init__(_bank_without_device(), 4, handle=_Weighted(), max_feed_samples=0)
    b = _bank_without_device(cap=320)
    ok = [np.zeros(320, np.int16), np.zeros(0, np.int16), np.zeros(5, np.int16), np.zeros(160, np.int16)]
    for bad in (ok[:3], ok + [ok[0]], ok[:3] + [np.zeros(321, np.int16)], ok[:3] + [np.zeros((2, 10), np.int16)]):
        with pytest.raises(ValueError):
            b.feed_samples(bad)
        with pytest.raises(ValueError):
            b.feed_samples(bad, want_logits=True)
    with pytest.raises(RuntimeError):                # speech is off
        b.feed_samples_speech(ok)
    b = _bank_without_device(cap=320, delay_rows=3)
    with pytest.raises(ValueError):
        b.feed_samples_speech(ok[:3] + [np.zeros(400, np.int16)])
    for call in (lambda: b.feed(np.zeros((4, 160), np.int16)), lambda: b.feed_speech(np.zeros((4, 160), np.int16)),
                 b.feed_pinned):                     # the fixed feeds on a ragged bank
        with pytest.raises(RuntimeError):
            call()
    fixed = _bank_without_device()
    with pytest.raises(RuntimeError):                # feed_samples on a fixed bank
        fixed.feed_samples(ok)
    fixed = _bank_without_device(delay_rows=3)
    with pytest.raises(RuntimeError):
        fixed.feed_samples_speech(ok)


class _Weighted(object):
    """A handle with weights and no device: StreamBank's cap check runs before the bank is created."""
    has_ffn = True

    def __getattr__(self, name):
        raise AssertionError("device work before the argument check: " + name)
