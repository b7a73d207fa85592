"""float64 oracle of the 16 kHz resampling path (include/vadb200.h, DESIGN.md section 5.8): the sample-format mapping
to int16 units, the channel mean, and scipy.signal.resample_poly, which the resampler's definition restates."""
from math import gcd

import numpy as np
from scipy.signal import firwin, resample_poly

OUT_RATE = 16000


def ratio(rate):
    """(up, down) for ``rate`` -> 16 kHz, or None when the rate is not accepted."""
    rate = int(rate)
    if rate < 4000 or rate > 384000:
        return None
    g = gcd(rate, OUT_RATE)
    up, down = OUT_RATE // g, rate // g
    return (up, down) if max(up, down) <= 1024 else None


def taps(rate):
    """firwin(2 half + 1, 1 / max(up, down), window=('kaiser', 5.0)) * up; the identity is one tap of 1."""
    up, down = ratio(rate)
    if up == down == 1:
        return np.ones(1)
    mx = max(up, down)
    return firwin(2 * 10 * mx + 1, 1.0 / mx, window=("kaiser", 5.0)) * up


def to_units(samples, fmt):
    """Samples as a file holds them -> float64 in int16 units (fmt: 'u8', 's16', 's24' (int32 of the 24-bit value),
    's32', 'f32', 'f64'); non-finite floats become 0."""
    x = np.asarray(samples)
    if fmt == "u8":
        return (x.astype(np.float64) - 128.0) * 256.0
    if fmt == "s16":
        return x.astype(np.float64)
    if fmt == "s24":
        return x.astype(np.float64) / 256.0
    if fmt == "s32":
        return x.astype(np.float64) / 65536.0
    v = x.astype(np.float64)
    return np.where(np.isfinite(v), v * 32768.0, 0.0)


def downmix(frames):
    """[n, C] (or [n]) int16-unit samples -> their channel mean."""
    f = np.asarray(frames, dtype=np.float64)
    return f if f.ndim == 1 else f.mean(axis=1)


def resample_exact(x, rate):
    """float64 resample_poly(x, up, down) of int16-unit samples (the identity at 16 kHz)."""
    up, down = ratio(rate)
    x = np.asarray(x, dtype=np.float64)
    if up == down == 1 or x.size == 0:
        return x.copy()
    return resample_poly(x, up, down)


def direct(x, rate):
    """The definition term by term: y[m] = sum_k x[k] h[m down + half - k up] (small inputs; checks resample_poly)."""
    up, down = ratio(rate)
    h = taps(rate)
    half = (h.size - 1) // 2
    x = np.asarray(x, dtype=np.float64)
    n_out = -(-x.size * up // down)
    y = np.zeros(n_out)
    for m in range(n_out):
        for k in range(x.size):
            j = m * down + half - k * up
            if 0 <= j < h.size:
                y[m] += x[k] * h[j]
    return y


def to_int16(y):
    """Round half to even, saturate."""
    return np.clip(np.rint(np.asarray(y, dtype=np.float64)), -32768, 32767).astype(np.int16)
