"""CPU: the 16 kHz resampler's definition (taps, lengths, accepted rates), the WAV format reader, argument checks of
the decode / resample entry points, and the float64 oracle against scipy."""
import ctypes as C
import struct

import numpy as np
import pytest
from scipy.io import wavfile
from scipy.signal import firwin, resample_poly

from oracle import ref_resample as rr

RATES = [8000, 11025, 16000, 22050, 24000, 32000, 44100, 48000, 96000]


@pytest.fixture(scope="module")
def lib():
    from vad_b200 import build, _lib
    build.build()
    return _lib.load()


@pytest.mark.parametrize("rate", RATES)
def test_taps_equal_scipy_firwin(lib, rate):
    n = lib.vadb200_resample_taps(rate, None)
    got = np.empty(n, dtype=np.float64)
    assert lib.vadb200_resample_taps(rate, got.ctypes.data_as(C.c_void_p)) == n
    up, down = rr.ratio(rate)
    if rate == 16000:
        assert n == 1 and got[0] == 1.0
        return
    mx = max(up, down)
    want = firwin(2 * 10 * mx + 1, 1.0 / mx, window=("kaiser", 5.0)) * up
    assert got.shape == want.shape
    assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))


def _primes(limit):
    sieve = np.ones(limit + 1, dtype=bool)
    sieve[:2] = False
    for p in range(2, int(limit ** 0.5) + 1):
        if sieve[p]:
            sieve[p * p::p] = False
    return np.flatnonzero(sieve)


@pytest.mark.parametrize("rate", RATES)
def test_resampled_length_equals_resample_poly(lib, rate):
    up, down = rr.ratio(rate)
    pr = _primes(10 ** 6)
    lengths = sorted({0, 1, 2, up, down} | set(int(p) for p in pr[::9000]) | {int(pr[-1])})
    for n in lengths:
        want = 0 if n == 0 else (n if rate == 16000 else len(resample_poly(np.zeros(n), up, down)))
        assert lib.vadb200_resampled_length(n, rate) == want, (rate, n)
    assert lib.vadb200_resampled_length(-1, rate) == -1


@pytest.mark.parametrize("rate", [44099, 3999, 0, -1, 384001, 4001])
def test_unsupported_rates_rejected(lib, rate):
    assert rr.ratio(rate) is None
    assert lib.vadb200_resampled_length(100, rate) == -1
    assert lib.vadb200_resample_taps(rate, None) == -1
    r = C.c_void_p()
    assert lib.vadb200_resampler_create(None, rate, C.byref(r)) == -2 and not r.value


def test_largest_accepted_ratio(lib):
    # 131072 Hz: up 125, down 1024 -- the longest filter the library accepts (20 481 taps)
    assert rr.ratio(131072) == (125, 1024)
    assert lib.vadb200_resample_taps(131072, None) == 20481
    assert lib.vadb200_resampled_length(1024, 131072) == 125


def test_entry_points_reject_bad_arguments_without_a_device(lib):
    raw = (C.c_uint8 * 64)()
    base = C.addressof(raw)
    odd = C.c_void_p(base + 1)
    dst = C.c_void_p(base)
    ln = C.c_void_p(base)
    for fmt in (0, 3, 4, 5):     # s16, s32, f32, f64 need an aligned stream
        assert lib.vadb200_decode_pcm(None, odd, fmt, 1, 0, ln, ln, ln, 1, 1, dst, None) == -1
        assert b"aligned" in lib.vadb200_last_error()
    assert lib.vadb200_decode_pcm(None, dst, 6, 1, 0, ln, ln, ln, 1, 1, dst, None) == -1
    assert lib.vadb200_decode_pcm(None, dst, 0, 0, 0, ln, ln, ln, 1, 1, dst, None) == -1
    assert lib.vadb200_decode_pcm(None, dst, 0, 33, 0, ln, ln, ln, 1, 1, dst, None) == -1
    assert lib.vadb200_decode_pcm(None, dst, 0, 1, 0, ln, ln, ln, 65536, 1, dst, None) == -1
    assert lib.vadb200_decode_pcm(None, dst, 1, 1, 0, ln, ln, ln, 1, 1, dst, None) == -1   # null handle
    offs = np.zeros(2, dtype=np.int64)
    assert lib.vadb200_resample_packed(None, 0, dst, offs.ctypes.data_as(C.c_void_p), offs.ctypes.data_as(C.c_void_p),
                                       1, dst, 64, offs.ctypes.data_as(C.c_void_p), dst, 64, None) == -1
    assert lib.vadb200_resample_workspace_bytes(None, 4) == -1
    assert lib.vadb200_resampler_create(None, 48000, None) == -1
    r = C.c_void_p()
    assert lib.vadb200_resampler_create(None, 48000, C.byref(r)) == -1 and not r.value
    assert lib.vadb200_resampler_destroy(None) == 0


# ---- wav_format against scipy.io.wavfile ---------------------------------------------------------------------
def _samples(code, n, ch, seed):
    rng = np.random.default_rng(seed)
    if code == 1:
        return rng.integers(0, 256, (n, ch)).astype(np.uint8)
    if code == 0:
        return rng.integers(-32768, 32768, (n, ch)).astype(np.int16)
    if code == 3:
        return rng.integers(-2 ** 31, 2 ** 31, (n, ch)).astype(np.int32)
    if code == 4:
        return rng.uniform(-1, 1, (n, ch)).astype(np.float32)
    return rng.uniform(-1, 1, (n, ch)).astype(np.float64)


def _hand_wav(path, rate, ch, bits, tag, payload, extensible=False):
    """RIFF/WAVE with a PCM (tag 1) or float (tag 3) payload, as plain WAVEFORMAT or WAVE_FORMAT_EXTENSIBLE, with an
    unrelated chunk before the data."""
    ba = ch * bits // 8
    if extensible:
        guid = struct.pack("<H", tag) + b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"
        fmt = struct.pack("<HHIIHHHHI", 0xFFFE, ch, rate, rate * ba, ba, bits, 22, bits, 0) + guid
    else:
        fmt = struct.pack("<HHIIHH", tag, ch, rate, rate * ba, ba, bits)
    junk = b"LIST" + struct.pack("<I", 5) + b"abcde\x00"
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + junk + b"data" + struct.pack("<I", len(payload)) \
        + payload + (b"\x00" if len(payload) & 1 else b"")
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def _s24_bytes(v):
    b = v.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3]
    return b.tobytes()


@pytest.mark.parametrize("ch", [1, 2, 6])
@pytest.mark.parametrize("code", [0, 1, 2, 3, 4, 5])
@pytest.mark.parametrize("extensible", [False, True])
def test_wav_format_agrees_with_scipy(tmp_path, code, ch, extensible):
    from vad_b200 import io
    n, rate = 1001, [8000, 11025, 22050, 44100, 48000, 96000][code]
    path = str(tmp_path / "a.wav")
    if code == 2:
        v = np.random.default_rng(code).integers(-2 ** 23, 2 ** 23, (n, ch)).astype(np.int32)
        _hand_wav(path, rate, ch, 24, 1, _s24_bytes(v.reshape(-1)), extensible)
    else:
        v = _samples(code, n, ch, code)
        if extensible:
            bits = v.dtype.itemsize * 8
            _hand_wav(path, rate, ch, bits, 3 if code in (4, 5) else 1, v.astype(v.dtype.newbyteorder("<")).tobytes(),
                      True)
        else:
            wavfile.write(path, rate, v if ch > 1 else v[:, 0])
    r, off, frames, channels, fmt = io.wav_format(path)
    srate, data = wavfile.read(path)
    data = data.reshape(len(data), -1)
    assert (r, frames, channels, fmt) == (srate, data.shape[0], data.shape[1], code)
    bps = {0: 2, 1: 1, 2: 3, 3: 4, 4: 4, 5: 8}[code]
    raw = np.fromfile(path, dtype=np.uint8, count=frames * channels * bps, offset=off)
    if code == 2:
        b = raw.reshape(-1, 3).astype(np.int32)
        mine = ((b[:, 0] << 8) | (b[:, 1] << 16) | (b[:, 2] << 24))     # scipy left-justifies 24-bit in int32
    else:
        mine = raw.view({0: "<i2", 1: "u1", 3: "<i4", 4: "<f4", 5: "<f8"}[code])
    assert np.array_equal(mine.reshape(data.shape), data)


def test_wav_layout_still_rejects_what_it_rejected(tmp_path):
    from vad_b200 import io
    path = str(tmp_path / "s.wav")
    wavfile.write(path, 16000, np.zeros((10, 2), dtype=np.int16))
    with pytest.raises(NotImplementedError):
        io.wav_layout(path)
    assert io.wav_format(path)[3] == 2


def test_wav_format_rejects_unknown_formats(tmp_path):
    from vad_b200 import io
    path = str(tmp_path / "alaw.wav")
    _hand_wav(path, 8000, 1, 8, 6, b"\x00" * 10)
    with pytest.raises(NotImplementedError):
        io.wav_format(path)


# ---- the oracle -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate", RATES)
def test_oracle_definition_is_resample_poly(rate):
    rng = np.random.default_rng(rate)
    for n in (0, 1, 7, 333):
        x = rng.integers(-32768, 32768, n).astype(np.float64)
        a, b = rr.resample_exact(x, rate), rr.direct(x, rate)
        assert a.shape == b.shape
        assert np.max(np.abs(a - b), initial=0.0) <= 1e-9


def test_oracle_format_mapping():
    assert np.array_equal(rr.to_units(np.array([0, 128, 255], dtype=np.uint8), "u8"), [-32768.0, 0.0, 32512.0])
    assert np.array_equal(rr.to_units(np.array([-2 ** 23, 256], dtype=np.int32), "s24"), [-32768.0, 1.0])
    assert np.array_equal(rr.to_units(np.array([-2 ** 31, 65536], dtype=np.int32), "s32"), [-32768.0, 1.0])
    assert np.array_equal(rr.to_units(np.array([1.0, np.nan, -np.inf], dtype=np.float32), "f32"), [32768.0, 0.0, 0.0])
    assert np.array_equal(rr.downmix([[1.0, 3.0], [2.0, 2.0]]), [2.0, 2.0])
    assert np.array_equal(rr.to_int16([0.5, 1.5, -2.5, 40000.0, -40000.0]), [0, 2, -2, 32767, -32768])
