"""CPU: the resampling ragged bank's index math (vad_b200/csrc/vad_stream_resample.h, driven on the host by
tests/emul/emul_stream_resample.cpp as the plan step and stream_resample_kernel use it).  For any chunking a stream's
per-feed output counts add up to M(N), the causal prefix of resample_poly that no later sample changes; no feed adds
more than cap16 and some feed adds exactly that; replaying the tiles' windows and the double-buffered history gives
the float64 oracle's outputs.  The Python surface rejects bad banks before any device work."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.signal import resample_poly

from oracle import ref_resample as rr
from test_gpu_resample import RATES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL = os.path.join(ROOT, "tests", "emul")
SO = os.path.join(EMUL, "libvademul_srs.so")
ALL = RATES + [16000]


@pytest.fixture(scope="module")
def emul():
    deps = [os.path.join(EMUL, "emul_stream_resample.cpp"),
            os.path.join(ROOT, "vad_b200", "csrc", "vad_stream_resample.h")]
    if not os.path.isfile(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", SO,
                               os.path.join(EMUL, "emul_stream_resample.cpp")])
    lib = C.CDLL(SO)
    lib.emul_srs_ready.restype = C.c_longlong
    lib.emul_srs_ready.argtypes = [C.c_longlong, C.c_int, C.c_int, C.c_int]
    lib.emul_srs_cap16.argtypes = [C.c_int] * 3
    lib.emul_srs_window_max.argtypes = [C.c_int] * 3
    lib.emul_srs_stream.restype = C.c_longlong
    lib.emul_srs_stream.argtypes = [C.c_int] * 6 + [C.c_void_p] * 7
    return lib


@pytest.fixture(scope="module")
def vlib():
    from vad_b200 import _lib, build
    build.build()
    return _lib.load()


def design(rate):
    up, down = rr.ratio(rate)
    half = 0 if up == down == 1 else 10 * max(up, down)
    K = (2 * half + 1 + up - 1) // up
    return up, down, half, K


def ready(n, rate):
    up, down, half, _ = design(rate)
    return 0 if n * up <= half else (n * up - 1 - half) // down + 1


def poly(rate):
    """Polyphase rows [up][K] of the float64 taps (row p: h[p], h[p + up], ...; zeros past the filter)."""
    up, _, _, K = design(rate)
    h = rr.taps(rate)
    t = np.zeros(up * K)
    t[:h.size] = h
    return np.ascontiguousarray(t.reshape(K, up).T)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def run(lib, rate, cap, sizes, signal):
    up, down, half, K = design(rate)
    sizes = np.ascontiguousarray(sizes, np.int32)
    signal = np.ascontiguousarray(signal, np.int16)
    tab = poly(rate)
    out = np.full(ready(len(signal), rate) + 1, np.nan)
    counts = np.full(len(sizes), -9, np.int32)
    tiles = np.full(len(sizes), -9, np.int32)
    widest = np.zeros(1, np.int32)
    m = lib.emul_srs_stream(up, down, half, K, cap, len(sizes), _p(sizes), _p(signal), _p(tab), _p(out), _p(counts),
                            _p(tiles), _p(widest))
    assert m >= 0
    return out[:m], counts, tiles, int(widest[0])


def chunkings(rate, rng):
    cap = rate // 25                                   # 40 ms packets at most
    up, down, _, K = design(rate)
    special = [0, 1, K - 1, K, K + 1, max(1, 160 * down // up), cap]
    a = [int(rng.choice(special)) if rng.random() < 0.5 else int(rng.integers(0, cap + 1)) for _ in range(60)]
    return cap, a


@pytest.mark.parametrize("rate", ALL)
def test_counts_add_up_to_the_ready_prefix(emul, vlib, rate):
    rng = np.random.default_rng(rate)
    up, down, half, K = design(rate)
    for _ in range(3):
        cap, sizes = chunkings(rate, rng)
        signal = rng.integers(-32768, 32768, sum(sizes)).astype(np.int16)
        _, counts, tiles, _ = run(emul, rate, cap, sizes, signal)
        cap16 = emul.emul_srs_cap16(cap, up, down)
        assert cap16 == -(-cap * up // down) <= 16000
        n = np.cumsum(sizes)
        assert np.array_equal(np.cumsum(counts), [ready(int(v), rate) for v in n])
        assert (counts <= cap16).all()
        assert np.array_equal(tiles, [0 if c == 0 else max(1, -(-int(k) // 256)) for c, k in zip(sizes, counts)])
        for v in n:
            assert emul.emul_srs_ready(int(v), up, down, half) == ready(int(v), rate)
            assert ready(int(v), rate) <= vlib.vadb200_resampled_length(int(v), rate)
    # the cap16 bound is tight: M(N + cap) - M(N) over one period of N (M(N + down) = M(N) + up) past the start
    for cap in (1, rate // 100, rate // 50, rate):
        cap16 = emul.emul_srs_cap16(cap, up, down)
        worst = max(ready(n + cap, rate) - ready(n, rate) for n in range(half + 1, half + 1 + down))
        assert worst == cap16, (cap, worst, cap16)


@pytest.mark.parametrize("rate", RATES)
def test_ready_prefix_is_what_scipy_gives_for_any_tail(rate):
    rng = np.random.default_rng(rate + 1)
    up, down, half, _ = design(rate)
    for n in (1, 7, half // up, half // up + 1, 500, 4410, 9999):
        x = rng.integers(-30000, 30000, n).astype(np.float64)
        tail = rng.integers(-30000, 30000, int(rng.integers(1, 3000))).astype(np.float64)
        m = ready(n, rate)
        a, b = resample_poly(x, up, down), resample_poly(np.r_[x, tail], up, down)
        assert m <= len(a)
        assert np.array_equal(a[:m], b[:m]), (n, m)


@pytest.mark.parametrize("rate", RATES)
def test_history_replay_reproduces_the_oracle(emul, rate):
    rng = np.random.default_rng(rate + 2)
    up, down, half, K = design(rate)
    cap, sizes = chunkings(rate, rng)
    sizes += [cap] * 3 + [0, 1, 2]
    signal = rng.integers(-32768, 32768, sum(sizes)).astype(np.int16)
    got, counts, _, widest = run(emul, rate, cap, sizes, signal)
    assert widest <= emul.emul_srs_window_max(up, down, K)
    ref = rr.resample_exact(signal, rate)[:len(got)]
    assert len(got) == ready(len(signal), rate)
    assert np.allclose(got, ref, rtol=0, atol=1e-7 * 32768 * np.abs(rr.taps(rate)).sum())


def test_bad_chunks_are_refused_by_the_replay(emul):
    with pytest.raises(AssertionError):
        run(emul, 48000, 480, [480, 481], np.zeros(961, np.int16))


@pytest.mark.parametrize("kw", [dict(sample_rate=8000),                             # a fixed bank at 8 kHz
                                dict(max_feed_samples=80, sample_rate=7),           # unsupported rates
                                dict(max_feed_samples=80, sample_rate=16001),
                                dict(max_feed_samples=0, sample_rate=8000),         # caps outside [1, r]
                                dict(max_feed_samples=8001, sample_rate=8000),
                                dict(max_feed_samples=48001, sample_rate=48000)])
def test_python_rejects_bad_banks_before_device_work(vlib, kw):
    from vad_b200.analyser import StreamBank
    with pytest.raises(ValueError):
        StreamBank(4, **kw)


def test_c_abi_rejects_without_a_device(vlib):
    out = C.c_void_p(123)
    assert vlib.vadb200_stream_bank_create_ragged_rate(None, 4, 480, 48000, C.byref(out)) == -1 and not out.value
    assert vlib.vadb200_stream_bank_create_ragged_rate(None, 4, 480, 48000, None) == -1
    assert vlib.vadb200_stream_bank_sample_rate(None) == -1
