"""Rounding bound of the 16 kHz resampler (tests/ only).

The kernel computes y32[m] = sum_i t_i * v_i for the taps t_i = fl32(h_i) of one polyphase row and the float32 input
v_i it staged, as a chain of K fused multiply-adds from 0 (K = ceil(len(h) / up) terms, zero taps included), then
rounds y32 half to even and saturates to int16.  Against y[m] = sum_i h_i x_i on the exact input x:

    |y32 - y| <= u sum |h_i| |x_i|                  (taps rounded to float32: |t_i - h_i| <= u |h_i|)
               + u / (1 - K u) sum_j |s_j|          (the FMA chain: step j rounds the partial sum
                                                     s_j = sum_{i <= j} t_i v_i, by at most u times its computed value)
               + sum |t_i| delta_i                  (input error |v_i - x_i| <= delta_i: decode, downmix)

with u = 2^-24.  The partial sums are taken in float64 in the kernel's tap order; the other two sums are resample_poly
of |x| or delta with |h| or |t| as the filter.  float64's own rounding (relative ~1e-15) is covered by the 1 % slack.
Where y lies farther than this bound beta_m from a rounding boundary (a half-integer) the int16 output is
round-half-even(saturate(y)) exactly; elsewhere it is within 1 LSB."""
import numpy as np
from scipy.signal import resample_poly

from oracle import ref_resample as rr

U = 2.0 ** -24


def _filter(x, h, up, down):
    """sum_k x[k] h[m down + half - k up] for a non-negative filter h of odd length 2 half + 1."""
    x = np.asarray(x, dtype=np.float64)
    if up == down == 1:
        return x * h[0]
    if x.size == 0:
        return np.zeros(0)
    return resample_poly(x, up, down, window=np.asarray(h, dtype=np.float64) / up)


def _chain(rate, v):
    """sum_j |s_j| per output: the partial sums of the kernel's tap loop y32 = fma(t_i, v_{kb - i}, y32), i = 0 .. K - 1."""
    up, down = rr.ratio(rate)
    h = rr.taps(rate)
    half = (h.size - 1) // 2
    K = -(-h.size // up)
    rows = np.zeros((up, K))
    for p in range(up):
        seg = h[p::up].astype(np.float32).astype(np.float64)
        rows[p, :seg.size] = seg
    n_out = -(-v.size * up // down)
    vp = np.concatenate([np.zeros(K), v, np.zeros(2)])
    out = np.empty(n_out)
    for m0 in range(0, n_out, 4096):
        m = np.arange(m0, min(n_out, m0 + 4096), dtype=np.int64)
        t = m * down + half
        kb = t // up
        idx = kb[:, None] - np.arange(K)[None, :] + K
        idx = np.clip(idx, 0, vp.size - 1)
        valid = (kb[:, None] - np.arange(K)[None, :] < v.size)
        terms = rows[t % up] * np.where(valid, vp[idx], 0.0)
        out[m0:m0 + m.size] = np.abs(np.cumsum(terms, axis=1)).sum(axis=1)
    return out, K


def beta(rate, x, v=None, delta=None):
    """Per-output bound on |y32 - y| for the exact input x (float64), the float32 input v the kernel read (default x)
    and the per-sample bound delta on |v - x| (default 0)."""
    up, down = rr.ratio(rate)
    h = rr.taps(rate)
    t = h.astype(np.float32).astype(np.float64)
    x = np.asarray(x, dtype=np.float64)
    v = x if v is None else np.asarray(v, dtype=np.float64)
    chain, K = _chain(rate, v)
    b = U * _filter(np.abs(x), np.abs(h), up, down) + U / (1.0 - K * U) * chain
    if delta is not None:
        b = b + _filter(np.broadcast_to(np.asarray(delta, dtype=np.float64), x.shape), np.abs(t), up, down)
    return b * 1.01 + 1e-300


def check(dev, rate, x, v=None, delta=None):
    """Asserts the rounding contract for one utterance; returns (outputs, outputs inside the band)."""
    dev = np.asarray(dev).astype(np.int64)
    y = rr.resample_exact(x, rate)
    assert dev.shape == y.shape, (dev.shape, y.shape)
    if y.size == 0:
        return 0, 0
    b = beta(rate, x, v, delta)
    target = rr.to_int16(y).astype(np.int64)
    frac = y - np.floor(y)
    band = np.abs(frac - 0.5) <= b
    bad = ~band & (dev != target)
    assert not bad.any(), "rate %d: %d outputs off the exact rounding, first at %d: dev %d want %d (y %.9f, beta %.3g)" % (
        rate, bad.sum(), np.flatnonzero(bad)[0], dev[bad][0], target[bad][0], y[bad][0], b[bad][0])
    far = band & (np.abs(dev - target) > 1)
    assert not far.any(), "rate %d: outputs more than 1 LSB off inside the band" % rate
    return int(y.size), int(band.sum())


def decode_delta(values, channels, exact_conversion):
    """Bound on |v - mean| for frames [n, C] of int16-unit values: float32 conversion (u |v_c| each unless exact),
    C - 1 float32 additions and one division."""
    a = np.abs(np.asarray(values, dtype=np.float64)).reshape(-1, channels)
    s = a.sum(axis=1)
    if channels == 1:
        return np.zeros(a.shape[0]) if exact_conversion else U * s * 1.01
    k = (channels - 1) + (0 if exact_conversion else 1) + 1
    return k * U / (1 - k * U) * s / channels * 1.01
