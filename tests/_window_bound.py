"""Window features on the kernel's own MFCC rows (tests/ only).

``window_check(c, feats, mode, path)`` takes the float32 MFCC rows ``c`` [T, 13] that MODE 0 writes for an utterance
and the feature rows [T - 5, 39] a kernel built from them (row r: centre t = r + 2, window c[t-2 .. t+2]), and checks:

* d1 = fl(c[t+1] - c[t-1]) bit for bit;
* dataset mode: z = c[t] and d2 = fl(fl(c[t+2] - c[t]) - fl(c[t] - c[t-2])) bit for bit;
* analyser mode: z and d2 within ``analyser_bound`` of float64 on the same float32 c; NaN in z and d2 exactly where
  the rule applies -- the five values bit-identical on the packed path (window_features_pairs: tensor-core block
  phases, dataset rows), ``==``-equal on the scalar one (window_features via classify_row: the fp32 block phase,
  windows_kernel, the stream bank);
* no inf anywhere, and every other entry finite.

``analyser_bound`` is first order over the kernel's operations (u = 2^-24): the four-add sum (gamma_4 sum |c|),
the product with 0.2f (its exact deviation from 0.2, and one rounding), the five differences (one rounding each;
a contracted FFMA rounds less), the FFMA chain of five squares (gamma_5) and its 0.2f product, rsqrtf (2 ulp:
relative 2^-22), the variance error through 1/sqrt, and the product d2 rsqrt.  The analyser d2 = (c4 - z) - (z - c0)
takes z's bound twice plus its three roundings."""
import numpy as np

U = 2.0 ** -24
F02 = float(np.float32(0.2))
MARGIN = 1.0 + 2.0 ** -9


def gamma(n):
    return n * U / (1 - n * U)


def windows(c):
    """[T - 5, 5, 13] float32 windows of the rows that have features (centres 2 .. T - 4)."""
    c = np.asarray(c, np.float32)
    T = c.shape[0]
    return np.stack([c[d:T - 5 + d] for d in range(5)], axis=1)


def analyser_bound(w):
    """(z_ref, z_bound, d2_ref, d2_bound) [n, 13] float64 for float32 windows w [n, 5, 13]; NaN refs where all five
    are equal (bound 0 there)."""
    c = np.asarray(w, np.float32).astype(np.float64)
    sabs = np.abs(c).sum(axis=1)
    s = c.sum(axis=1)
    mu = s / 5
    d = c - mu[:, None]
    var = (d * d).mean(axis=1)
    e_sum = gamma(4) * sabs
    e_mu = F02 * e_sum + abs(F02 - 0.2) * np.abs(s)
    e_mu += U * (np.abs(mu) + e_mu)
    e_d = e_mu[:, None] + U * (np.abs(d) + e_mu[:, None])
    Q = (d * d).sum(axis=1)
    e_Q = (2 * np.abs(d) * e_d + e_d * e_d).sum(axis=1)
    e_Q += gamma(5) * (Q + e_Q)
    e_var = F02 * e_Q + abs(F02 - 0.2) * (Q + e_Q)
    e_var += U * (var + e_var)
    with np.errstate(divide="ignore", invalid="ignore"):
        rel = e_var / var
        R = 1.0 / np.sqrt(var)
        ok = rel < 0.5
        relc = np.where(ok, rel, 0.0)
        e_R = np.where(ok, R * ((1.0 / np.sqrt(1 - relc) - 1) + 2.0 ** -22 / np.sqrt(1 - relc)), np.inf)
        z = d[:, 2] * R
        e_z = e_d[:, 2] * (R + e_R) + np.abs(d[:, 2]) * e_R
        e_z += U * (np.abs(z) + e_z)
        d2 = (c[:, 4] - z) - (z - c[:, 0])
        e_d2 = 2 * e_z + U * (np.abs(c[:, 4] - z) + e_z) + U * (np.abs(z - c[:, 0]) + e_z)
        e_d2 += U * (np.abs(d2) + 2 * e_d2)
    eq = var == 0
    z = np.where(eq, np.nan, z)
    d2 = np.where(eq, np.nan, d2)
    return z, np.where(eq, 0.0, e_z * MARGIN), d2, np.where(eq, 0.0, e_d2 * MARGIN)


def nan_rule(w, path):
    """[n, 13] bool: where the kernel must write NaN into z and d2 (analyser mode)."""
    w = np.asarray(w, np.float32)
    if path == "pairs":
        b = w.view(np.uint32)
        return np.all(b == b[:, :1], axis=1)
    return np.all(w == w[:, :1], axis=1)


def window_check(c, feats, mode, path):
    """Check feature rows against section 3's rules; returns {"z": worst |d| / bound, "d2": ...} (analyser) or {}."""
    w = windows(c)
    f = np.asarray(feats, np.float32)
    assert f.shape == (w.shape[0], 39), (f.shape, w.shape)
    assert not np.isinf(f).any(), "inf in a feature row"
    d1 = w[:, 3] - w[:, 1]
    assert np.array_equal(f[:, 13:26].view(np.uint32), d1.view(np.uint32)), "d1 differs from fl(c[t+1] - c[t-1])"
    if mode == "dataset":
        d2 = (w[:, 4] - w[:, 2]) - (w[:, 2] - w[:, 0])
        assert np.array_equal(f[:, :13].view(np.uint32), w[:, 2].view(np.uint32)), "dataset c differs"
        assert np.array_equal(f[:, 26:].view(np.uint32), d2.view(np.uint32)), "dataset d2 differs"
        return {}
    nan = nan_rule(w, path)
    for g, name in ((0, "z"), (2, "d2")):
        got = f[:, 13 * g:13 * (g + 1)]
        assert np.array_equal(np.isnan(got), nan), "%s: NaN where the rule does not put one (or none where it does)" \
            % name
    zr, zb, dr, db = analyser_bound(w)
    out = {}
    for g, name, ref, bnd in ((0, "z", zr, zb), (2, "d2", dr, db)):
        got = f[:, 13 * g:13 * (g + 1)].astype(np.float64)
        m = ~nan
        err = np.abs(got[m] - ref[m])
        bad = ~(err <= bnd[m])
        assert not bad.any(), "%s: %d entries exceed the bound (worst |d| / bound %.3g)" % (
            name, bad.sum(), np.max(err / bnd[m]))
        with np.errstate(invalid="ignore", divide="ignore"):
            fr = np.where(bnd[m] > 0, err / bnd[m], 0.0)
        out[name] = float(fr.max()) if fr.size else 0.0
    return out
