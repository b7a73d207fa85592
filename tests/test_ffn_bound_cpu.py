"""CPU: the per-entry logit bound of tests/_ffn_bound.py against numpy emulations of each device FFN scheme.

The emulations follow the kernels' arithmetic step by step: ffn_forward's FFMA order (fp32), ffn_tc_tile's tf32
hi/lo split (tc), and ffn_tc16_tile's fp16 hi/lo scheme (tc16: layer 1 on one accumulator, layers 2-4 on the 2N
scheme) on the very blob tc16_pack_weights packs (read back through tests/emul/emul_ffn.cpp and de-swizzled with
tc16_pack_layer's index formula).  Each tensor-core instruction's sum is truncated to fp32, the accumulation the
bound assumes.  Every faithful emulation stays within a quarter of the bound; every
mutant -- a product dropped in one layer, a subnormal lo flushed, a scale off by two, an unscaled bias, a shifted
layer-1 column -- exceeds it at least five-fold somewhere."""
import numpy as np
import pytest

from oracle import ref_math as rm
from vad_b200.synth import synth_utterance

import _ffn_bound as fb

SETS = fb.weight_sets()
MUTANT_SETS = ["glorot0", "glorot_x3_bias", "trained"]


# ---- emulation helpers -----------------------------------------------------------------------------------------------
def f32(v):
    return np.asarray(v, np.float64).astype(np.float32)


def rz32(v):
    """float64 -> float32 toward zero."""
    v = np.asarray(v, np.float64)
    f = v.astype(np.float32)
    over = np.abs(f.astype(np.float64)) > np.abs(v)
    f[over] = np.nextafter(f[over], np.float32(0))
    return f


def split16(a, flush_subnormal_lo=False):
    """tc16_split2: fp16 hi to nearest, lo = fp16(a - hi) (the residual is exact in fp32)."""
    a = f32(a)
    hi = a.astype(np.float16)
    lo = (a - hi.astype(np.float32)).astype(np.float16)
    if flush_subnormal_lo:
        lo = np.where(np.abs(lo.astype(np.float32)) < 2.0 ** -14, np.float16(0), lo)
    return hi.astype(np.float64), lo.astype(np.float64)


def tf32(a):
    """tf32 operand of an fp32 register: the top 19 bits (tc_split, tf32_hi)."""
    u = f32(a).view(np.uint32) & np.uint32(0xFFFFE000)
    return u.view(np.float32)


def tc_feat_col(f):
    g, k = f // 13, f % 13
    q, e = k // 2, k % 2
    return 6 * q + 2 * g + e if q < 4 else 24 + 6 * (q - 4) + 2 * g + e


def layer1_columns(x, shift=0):
    """[n, 48] layer-1 A operand: feature f in column tc_feat_col(f) (shift: feature f where f + shift belongs)."""
    x = f32(x)
    a = np.zeros((x.shape[0], fb.K_PAD[0]), np.float32)
    for f in range(39):
        a[:, tc_feat_col((f + shift) % 39)] = x[:, f]
    return a


def unpack(blob, l, fp16):
    """(B_hi, B_lo) [K, N] of layer l from the packed blob (tc16_pack_layer / tc_pack_layer index formulas)."""
    K, N = fb.K_PAD[l], fb.N_PAD[l]
    off = sum(2 * fb.K_PAD[i] * fb.N_PAD[i] for i in range(l))
    k, n = np.meshgrid(np.arange(K), np.arange(N), indexing="ij")
    if fp16:
        ihi = ((k // 8) * (2 * N // 8) + n // 8) * 64 + (n % 8) * 8 + k % 8
        ilo = ((k // 8) * (2 * N // 8) + (N + n) // 8) * 64 + ((N + n) % 8) * 8 + k % 8
        v = blob.view(np.float16)
    else:
        ihi = ((k // 4) * (2 * N // 8) + n // 8) * 32 + (n % 8) * 4 + k % 4
        ilo = ((k // 4) * (2 * N // 8) + (N + n) // 8) * 32 + ((N + n) % 8) * 4 + k % 4
        v = blob
    return v[off + ihi].astype(np.float64), v[off + ilo].astype(np.float64)


def mma_chain(acc, terms, g):
    """Accumulate a list of (A [n, K], B [K, N]) products one g-deep instruction at a time, k-step major, in the
    listed order within a k-step; each instruction's exact sum is truncated to fp32."""
    K = terms[0][0].shape[1]
    for j in range(0, K, g):
        for a, b in terms:
            acc = rz32(acc.astype(np.float64) + a[:, j:j + g] @ b[j:j + g])
    return acc


# ---- the emulated schemes -------------------------------------------------------------------------------------------
def emul_fp32(x, w):
    """ffn_forward: per output, the bias then one FFMA per input, in input order."""
    h = f32(x)
    for l in range(4):
        W, b = f32(w["W%d" % (l + 1)]), f32(w["b%d" % (l + 1)])
        z = np.broadcast_to(b, (h.shape[0], W.shape[1])).astype(np.float32)
        for i in range(W.shape[0]):
            z = f32(h[:, i:i + 1].astype(np.float64) * W[i].astype(np.float64) + z)
        h = np.maximum(z, np.float32(0)) if l < 3 else z
    return h.astype(np.float64)


def emul_tc(x, w, pk):
    """ffn_tc_tile: tf32 hi/lo, D[0:N] += a_hi B_hi, a_lo B_hi; D[N:2N] += a_hi B_lo; 8 products per instruction."""
    a = layer1_columns(x)
    for l in range(4):
        N, n_out = fb.N_PAD[l], np.asarray(w["b%d" % (l + 1)]).size
        bh, bl = unpack(pk["blob32"], l, False)
        bl = tf32(bl).astype(np.float64)
        ah = tf32(a).astype(np.float64)
        al = tf32(f32(a) - tf32(a)).astype(np.float64)
        zero = np.zeros((a.shape[0], N), np.float32)
        v = mma_chain(zero, [(ah, bh), (al, bh)], 8)
        u = mma_chain(zero, [(ah, bl)], 8)
        b = np.zeros(N, np.float32)
        b[:n_out] = w["b%d" % (l + 1)]
        z = f32(f32(v.astype(np.float64) + u).astype(np.float64) + b)
        if l == 3:
            return z[:, :3].astype(np.float64)
        a = np.maximum(z, np.float32(0))


def emul_tc16(x, w, pk, drop=None, flush_lo=False, pre2=None, post2=None, bias_unscaled=False, shift=0):
    """ffn_tc16_tile.  Mutations: drop = (layer, "hh" | "hl" | "lh");
    flush_lo: subnormal lo halves of the activations become 0; pre2 / post2 = layer whose activation pre-scale /
    weight post-scale is doubled; bias_unscaled: c_l = b_l; shift: layer-1 features one column off."""
    postp = f32(pk["postp"]).copy()
    post3 = np.float32(pk["post"][3])
    cs = [f32(c).copy() for c in pk["c"]]
    if bias_unscaled:
        cs = [f32(w["b%d" % (l + 1)]) for l in range(3)]
    a = layer1_columns(x, shift)
    if pre2 is not None:
        if pre2 == 0:
            a = a * np.float32(2)
        else:
            postp[pre2 - 1] *= 2
            cs[pre2 - 1] = cs[pre2 - 1] * np.float32(2)
    if post2 is not None:
        if post2 == 3:
            post3 = post3 * np.float32(2)
        else:
            postp[post2] *= 2
    for l in range(4):
        N = fb.N_PAD[l]
        bh, bl = unpack(pk["blob16"], l, True)
        ah, al = split16(a, flush_lo)
        prods = {"hh": (ah, bh), "hl": (ah, bl), "lh": (al, bh)}
        live = [p for p in ("hh", "hl", "lh") if drop != (l, p)]
        zero = np.zeros((a.shape[0], N), np.float32)
        if l == 0:
            d = mma_chain(zero, [prods[p] for p in live], 16)
        else:
            v = mma_chain(zero, [prods[p] for p in live if p != "hl"], 16)
            u = mma_chain(zero, [prods[p] for p in live if p == "hl"], 16) if "hl" in live else zero
            d = f32(v.astype(np.float64) + u)
        if l == 3:
            return f32(d[:, :3].astype(np.float64) * post3 + f32(w["b4"])).astype(np.float64)
        a = np.maximum(f32(d.astype(np.float64) * postp[l] + cs[l]), np.float32(0))


def emulate(impl, x, w, pk):
    if impl == "fp32":
        return emul_fp32(x, w)
    if impl == "tc":
        return emul_tc(x, w, pk)
    return emul_tc16(x, w, pk)


# ---- test rows ------------------------------------------------------------------------------------------------------
def bound_rows():
    """Analyser feature rows of three utterances (one of them quiet), N(0, 1) and N(0, 30) rows, rows at +-the feature
    bounds, all-zero and -0 rows, tiny rows (|x| ~ 1e-3: layer 1's lo halves subnormal) and rows of magnitude ~ 2^-3
    whose lo halves are subnormal with the largest residuals."""
    rng = np.random.default_rng(17)
    utts = [synth_utterance(7, 0, 16000 * 3), synth_utterance(7, 1, 16000 * 2), synth_utterance(8, 0, 16000 * 2) // 300]
    feats = np.concatenate([rm.vad_utterance(u, rm.glorot_ffn(0))[1] for u in utts])
    feats = feats[np.isfinite(feats).all(axis=1)]
    bound = fb.FEAT_BOUND
    rows = [feats, rng.standard_normal((400, 39)), rng.standard_normal((200, 39)) * 30,
            np.where(rng.random((64, 39)) < 0.5, -1, 1) * bound * rng.integers(0, 2, (64, 39)),
            np.zeros((2, 39)), -np.zeros((2, 39)),
            rng.standard_normal((200, 39)) * 1e-3,
            rng.choice([-1, 1], (200, 39)) * rng.uniform(2.0 ** -4, 2.0 ** -2, (200, 39))]
    return np.concatenate(rows).astype(np.float32)


ROWS = bound_rows()
_CACHE = {}


def bound_of(name, impl):
    k = (name, impl)
    if k not in _CACHE:
        _CACHE[k] = fb.ffn_bound(ROWS, SETS[name], impl)
    return _CACHE[k]


def impls_of(name):
    return fb.IMPLS if fb.tc16_scales(SETS[name])[0] else ("fp32", "tc")


# ---- tests ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(SETS))
def test_scales_restate_tc16_pack_weights(name):
    """tc16_scales (Python) chooses what tc16_pack_weights (C++) chooses; the folded constants follow from them."""
    w = SETS[name]
    ok, pre, post, sw = fb.tc16_scales(w)
    pk = fb.pack(w)
    assert ok == pk["ok"]
    if not ok:
        return
    assert np.array_equal(pk["pre"], f32(pre)) and np.array_equal(pk["post"], f32(post))
    assert np.array_equal(pk["postp"], f32(np.append(post[:3] * pre[1:], post[3])))
    for l in range(3):
        assert np.array_equal(pk["c"][l], f32(w["b%d" % (l + 1)]) * np.float32(pre[l + 1]))
    for l in range(4):                    # the blob holds the scaled weights split in fp16, at tc16_pack_layer's places
        bh, bl = unpack(pk["blob16"], l, True)
        W = np.asarray(w["W%d" % (l + 1)], np.float64)
        k_idx = [tc_feat_col(f) for f in range(39)] if l == 0 else list(range(W.shape[0]))
        sw_hi_lo = (bh + bl)[k_idx][:, :W.shape[1]]
        assert np.all(np.abs(sw_hi_lo - W * sw[l]) <= 2.0 ** -22 * np.abs(W * sw[l]) + 2.0 ** -25)


def test_deep_sets_straddle_the_fp16_range():
    assert max(-np.log2(fb.tc16_scales(SETS["deep_ea60"])[1])) == 60
    assert not fb.pack(SETS["beyond_ea61"])["ok"]


@pytest.mark.parametrize("name", list(SETS))
def test_faithful_emulations_within_a_quarter_of_the_bound(name):
    w = SETS[name]
    pk = fb.pack(w)
    ref = fb.forward64(ROWS, w)[0][3]
    for impl in impls_of(name):
        err = np.abs(emulate(impl, ROWS, w, pk) - ref)
        bound = bound_of(name, impl)
        assert np.all(err <= 0.25 * bound), "%s %s: worst |d| / bound %.3g" % (name, impl, np.max(err / bound))


def mutants():
    out = {}
    for l in range(4):
        for p in ("hh", "hl", "lh"):
            out["drop %s layer %d" % (p, l + 1)] = dict(drop=(l, p))
        out["pre x2 layer %d" % (l + 1)] = dict(pre2=l)
        out["post x2 layer %d" % (l + 1)] = dict(post2=l)
    out["subnormal lo flushed"] = dict(flush_lo=True)
    out["bias unscaled"] = dict(bias_unscaled=True)
    out["layer-1 columns shifted by one"] = dict(shift=1)
    return out


@pytest.mark.parametrize("name", MUTANT_SETS)
def test_mutants_exceed_the_bound_five_fold(name):
    """A kernel that loses a product, a lo half, a scale or a column is caught with a margin.  The unscaled-bias
    mutant computes the faithful function where every c_l equals b_l (zero biases, or pre[l+1] == 1 throughout) and
    is only required where it differs."""
    w = SETS[name]
    pk = fb.pack(w)
    ref = fb.forward64(ROWS, w)[0][3]
    bound = bound_of(name, "tc16")
    weak = {}
    for mname, kw in mutants().items():
        if mname == "bias unscaled" and all(np.array_equal(pk["c"][l], f32(w["b%d" % (l + 1)])) for l in range(3)):
            continue
        got = emul_tc16(ROWS, w, pk, **kw)
        worst = np.nanmax(np.abs(got - ref) / bound)
        if not worst >= 5.0:
            weak[mname] = worst
    assert not weak, weak


def test_relu_rule_keeps_error_of_units_just_below_zero():
    """A unit whose float64 pre-activation lies in (-e, 0] can come out positive on the device, so its error must
    pass on.  Built by hand: layer 1's unit 0 gets z = -2^-30 from a row whose rounding bound e is far larger; every
    other unit is off.  The bound keeps unit 0's error (logits bound > 0 from layer 1); the rule z > 0 of
    test_gpu_signals.rounding_reach drops it."""
    w = {k: np.zeros_like(v) for k, v in rm.glorot_ffn(0).items()}
    w["W1"][0, 0], w["W1"][1, 0] = 1.0, -1.0
    w["W2"][0, 0] = w["W3"][0, 0] = w["W4"][0, 0] = 1.0
    x = np.zeros((1, 39), np.float32)
    x[0, 0], x[0, 1] = 1.0, 1.0 + 2.0 ** -23          # z = -2^-23, while e_1 >= 2^-24 x 2 x (1 + 1)
    z1 = fb.forward64(x, w)[0][0][0, 0]
    assert -2.0 ** -22 < z1 < 0
    for impl in fb.IMPLS:
        assert fb.ffn_bound(x, w, impl)[0, 0] > 0, impl
    u = 2.0 ** -20                                     # rounding_reach's rule, restated
    h, e = x.astype(np.float64), np.zeros((1, 39))
    for i in (1, 2, 3, 4):
        Wi, bi = w["W%d" % i].astype(np.float64), w["b%d" % i].astype(np.float64)
        z = h @ Wi + bi
        e = e @ np.abs(Wi) + u * (np.abs(h) @ np.abs(Wi) + np.abs(bi))
        if i < 4:
            e = np.where(z > 0, e, 0.0)
            h = np.maximum(z, 0.0)
    assert e[0, 0] == 0.0
