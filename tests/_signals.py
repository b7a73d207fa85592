"""Deterministic signal catalogue (tests/ only): int16 utterances of about 1-2 s at 16 kHz that reach where
white Irwin-Hall noise (vad_b200/synth.py, about +-11k) never goes -- samples at and near the int16 rails, full-scale
tones and chirps whose mel bands differ by tens of dB, band-limited noise, LSB-level audio, signals whose frames are
bit-identical (sigma5 == 0 -> NaN analyser rows), and one utterance that switches between families mid-stream so
segment starts and frame boundaries fall inside full-scale regions.  Seeded numpy / scipy only."""
from collections import OrderedDict

import numpy as np
from scipy.signal import butter, sosfilt

FS = 16000
LO, HI = -32768, 32767


def _pcm(x):
    return np.clip(np.round(np.asarray(x, dtype=np.float64)), LO, HI).astype(np.int16)


def _t(n):
    return np.arange(n) / float(FS)


def clipped_noise(n, seed=1):
    """Gaussian noise with a full-scale standard deviation, clipped: about a third of the samples sit on a rail."""
    return _pcm(np.random.default_rng(seed).standard_normal(n) * 32768.0)


def square(n, period):
    """+-full scale square wave; period 2 alternates 32767 / -32768 (all energy in the Nyquist bin)."""
    k = np.arange(n) % period
    return np.where(k < period // 2, HI, LO).astype(np.int16)


def constant(n, value):
    return np.full(n, value, dtype=np.int16)


def tone(n, hz, amp=32767.0, phase=0.3):
    return _pcm(amp * np.sin(2 * np.pi * hz * _t(n) + phase))


def hop_periodic_tone(n):
    """Full-scale 100 Hz: its period is the 160-sample hop, so every frame is bit-identical (sigma5 == 0)."""
    return np.tile(tone(160, 100.0), n // 160 + 1)[:n]


def chirp(n, f0=50.0, f1=8000.0, amp=30000.0, dur=2.0):
    """Linear chirp from f0 at t = 0 to f1 at t = dur.  A faster sweep smears a frame's energy so far that the
    float32 FFT's rounding floor, in numpy's float32 path as in the kernels, reaches the MFCC tolerance in the
    lowest bands (1.5 s: 1.25x the tolerance at the 7 kHz frames); 2 s keeps a margin of about 5x."""
    t = _t(n)
    k = (f1 - f0) / dur
    return _pcm(amp * np.sin(2 * np.pi * (f0 * t + 0.5 * k * t * t)))


def tone_lsb_noise(n, seed=2):
    """440 Hz at 32000 plus uniform {-1, 0, 1} LSB noise."""
    rng = np.random.default_rng(seed)
    return _pcm(32000.0 * np.sin(2 * np.pi * 440.0 * _t(n)) + rng.integers(-1, 2, n))


def band_noise(n, hz, btype, seed, std=20000.0):
    """8th-order Butterworth low- / high-pass of white noise, scaled to ``std`` and clipped."""
    sos = butter(8, hz, btype=btype, fs=FS, output="sos")
    x = sosfilt(sos, np.random.default_rng(seed).standard_normal(n + 2000))[2000:]   # drop the filter's start-up
    return _pcm(x / x.std() * std)


def impulses(n, every=250, at=7):
    """32767 every ``every`` samples on digital silence.  Not every 400: then each frame holds exactly one impulse,
    every frame has the same magnitude spectrum in exact arithmetic, and whether the analyser's sigma5 comes out 0
    (a NaN row) is decided by rounding alone, in the float64 oracle as in the kernels."""
    x = np.zeros(n, dtype=np.int16)
    x[at::every] = HI
    return x


def lsb_square(n, half=3):
    return ((np.arange(n) // half) % 2).astype(np.int16)


def lsb_noise(n, seed=3):
    """Uniform noise in [-2, 2] LSB."""
    return np.random.default_rng(seed).integers(-2, 3, n).astype(np.int16)


def mixed(n, seed=4):
    """Families switched every 1 234 samples (not a multiple of the 160-sample hop), full-scale pieces first."""
    gens = [lambda m: clipped_noise(m, seed), lambda m: square(m, 2), lambda m: tone(m, 1000.0),
            lambda m: constant(m, LO), lambda m: lsb_noise(m, seed), lambda m: square(m, 74),
            lambda m: constant(m, HI), lambda m: impulses(m)]
    piece = 1234
    out = [gens[i % len(gens)](piece) for i in range((n + piece - 1) // piece)]
    return np.concatenate(out)[:n]


# Signals whose spectrum, once pre-emphasised (0.97) and Hamming-windowed, spans more dynamic range than float32
# resolves at the MFCC tolerance: the window's low leakage leaves mel bands 100 dB and more below the peak, where the
# FFT's float32 rounding floor dominates.  A float32 restatement of the front end (numpy, as the reference's own
# float32 path computes it) misses the tolerance on each of them, so no float32 kernel can be held to it there.
# The front-end tests still run them through every batch; test_signals_cpu.py checks that each stays beyond float32.
WINDOWED_FLOAT32_FLOOR = ("chirp_50_8k", "tone_440_lsb_noise", "lowpass_300_noise", "highpass_7k_noise")


def catalogue():
    """name -> int16 PCM.  Lengths differ (a ragged batch), 1.0-2.0 s; the mixed utterance is 3 s so it spans several
    64-frame segments."""
    specs = [
        ("clipped_noise", lambda n: clipped_noise(n)),
        ("square_p74", lambda n: square(n, 74)),
        ("square_nyquist", lambda n: square(n, 2)),
        ("dc_min", lambda n: constant(n, LO)),
        ("dc_max", lambda n: constant(n, HI)),
        ("tone_200", lambda n: tone(n, 200.0)),
        ("tone_1k", lambda n: tone(n, 1000.0)),
        ("tone_7900", lambda n: tone(n, 7900.0)),
        ("tone_100_hop_periodic", hop_periodic_tone),
        ("chirp_50_8k", lambda n: chirp(32000 + 17)),
        ("tone_440_lsb_noise", lambda n: tone_lsb_noise(n)),
        ("lowpass_300_noise", lambda n: band_noise(n, 300.0, "lowpass", 5)),
        ("highpass_7k_noise", lambda n: band_noise(n, 7000.0, "highpass", 6)),
        ("impulse_train", lambda n: impulses(n)),
        ("lsb_square", lambda n: lsb_square(n)),
        ("lsb_noise", lambda n: lsb_noise(n)),
    ]
    out = OrderedDict()
    for i, (name, gen) in enumerate(specs):
        out[name] = gen(16000 + 1013 * i)
    out["mixed"] = mixed(48000 + 77)
    return out
