"""Per-entry rounding bound of the classifier's logits (tests/ only).

``ffn_bound(x, w, impl)`` bounds |logit_device - logit_float64| for the 39-64-32-16-3 FFN evaluated on the exact
float32 rows ``x`` by one device implementation.  Feature error plays no part: the reference is the float64 forward
pass of the same float32 inputs the kernel used.  The bound is carried layer by layer: the error e of a layer's inputs
passes on through |W|, and each layer adds its own rounding, computed from absolute values:

    e_z = |W|^T e + d,   d = u_prod |W|^T H + acc + epilogue + floors,   H = |h| + e (a bound on the device's |h|)

ReLU is 1-Lipschitz, so e passes through it, except for units whose float64 pre-activation is <= -e_z: the device's
pre-activation is then <= 0 as well and the unit is exactly 0 on both sides.  That absolute-value recursion decides
which units are surely on, surely off or either; the bound returned carries each layer's own rounding d_l to the
logits through the signed later layers instead (interval Jacobians, see the end of ffn_bound), which keeps the
cancellation |W| loses.

Per implementation (u = 2^-24, the fp32 unit roundoff):

* ``fp32`` (vad_core.cuh ffn_forward): a chain of K FFMAs from the bias, each rounded to nearest:
  d <= gamma_K (|b| + |W|^T H), gamma_K = K u / (1 - K u).
* ``tc`` (ffn_tc_tile, tf32 hi/lo): x = x_hi + x_lo with x_hi the top 11 significant bits (truncation) and x_lo read
  by the tensor core as tf32, i.e. truncated to 11 bits, which loses the 2 lowest bits of x (< 2^-21 |x|); the
  dropped x_lo w_lo is < 2^-20 |x w|.  Per product: u_prod = 2^-20 + 2 x 2^-21 = 2^-19.
* ``tc16`` (ffn_tc16_tile: layer 1 on one accumulator, layers 2-4 on the 2N scheme): operands a = h pre[l] and
  w sw_l, split to nearest in fp16.  Each split half errs by at most 2^-11 of
  what it rounds, or by half the fp16 subnormal spacing (2^-25) where it is subnormal, so a - a_hi - a_lo is within
  2^-22 |a| + 2^-25, and the dropped a_lo w_lo adds 2^-22 |a w|.  Per product, in unscaled units:
  3 x 2^-22 |h w| + 2^-25 (|w| / pre[l] + |h| / sw_l).  The scales are the ones tc16_pack_weights chooses
  (``tc16_scales`` restates it; the CPU suite checks the restatement against the C++).

Accumulation (tensor-core paths).  Products of tf32 or fp16 operands are exact in fp32.  How tcgen05 rounds the fp32
sum has not been measured, so each MMA instruction (8 tf32 or 16 fp16 products plus the accumulator) is taken to
truncate its result to fp32 once, toward zero: an error below 2 u |partial sum| <= 2 u |W|^T H.  A layer's output
sees one such rounding per instruction that accumulates into its column: 2 K/g on the 2N scheme (a_hi B_hi and
a_lo B_hi share the first N columns; a_hi B_lo goes to the second N, whose sum is below 2^-9 of the first), 3 K/g on
the single accumulator of tc16's layer 1.  K is the padded depth (48, 64, 32, 16).  The epilogue adds the two
halves and the bias (tc) or runs one FFMA with the folded constants (tc16), each rounded to nearest: 2 u (|W|^T H +
|b|).  Everything above is first order; the constants carry a 2^-9 margin for the second-order terms.
"""
import ctypes as C
import math
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL = os.path.join(ROOT, "tests", "emul")
FFN_KEYS = ("W1", "b1", "W2", "b2", "W3", "b3", "W4", "b4")
K_PAD = (48, 64, 32, 16)       # kTcK1 .. kTcK4
N_PAD = (64, 32, 16, 16)       # kTcN1 .. kTcN4
FEAT_BOUND = np.repeat([1353.0, 2706.0, 5416.0], 13)   # kFeatBoundZ / D1 / D2 (ffn_tc.cuh)
IMPLS = ("fp32", "tc", "tc16")
U = 2.0 ** -24
MARGIN = 1.0 + 2.0 ** -9


def flat_weights(w):
    return np.concatenate([np.asarray(w[k], np.float32).ravel() for k in FFN_KEYS]).astype(np.float32)


# ---- tc16_pack_weights (ffn_tc.cuh) restated -----------------------------------------------------------------------
def tc16_scales(w):
    """(ok, pre[4], post[4], sw[4]) as tc16_pack_weights chooses them; ok False where it keeps the tf32 path."""
    bound = [float(b) for b in FEAT_BOUND]
    pre, post, sw = [], [], []
    for l in range(4):
        W = np.asarray(w["W%d" % (l + 1)], np.float32).astype(np.float64)
        b = np.asarray(w["b%d" % (l + 1)], np.float32).astype(np.float64)
        amax = max(bound)
        wmax = float(np.abs(W).max())
        if not (amax < 1e30 and wmax < 1e30):
            return False, None, None, None
        ea = int(math.ceil(math.log2(amax / 32000.0))) if amax > 32000.0 else 0
        ew = int(math.floor(math.log2(16000.0 / wmax))) if wmax > 0.0 else 0
        if ea > 60 or ew > 60 or ew < -60 or (l == 0 and ea != 0):
            return False, None, None, None
        pre.append(2.0 ** -ea)
        post.append(2.0 ** (ea - ew))
        sw.append(2.0 ** ew)
        nb = []
        Wa = np.abs(W)
        for j in range(W.shape[1]):      # the C++ order: |b_j| then sum_i |W_ij| bound_i, sequentially in double
            s = abs(float(b[j]))
            for i in range(W.shape[0]):
                s += float(Wa[i, j]) * bound[i]
            nb.append(s)
        bound = nb
    return True, np.array(pre), np.array(post), np.array(sw)


# ---- the C++ packing itself, through tests/emul/emul_ffn.cpp ------------------------------------------------------
_SHIM = []


def shim():
    """ctypes handle of tests/emul/emul_ffn.cpp, built with g++ against the CUDA headers next to the nvcc that
    vad_b200.build uses (cuda_fp16.h)."""
    if _SHIM:
        return _SHIM[0]
    src = os.path.join(EMUL, "emul_ffn.cpp")
    so = os.path.join(EMUL, "libvademul_ffn.so")
    deps = [src] + [os.path.join(ROOT, "vad_b200", "csrc", f) for f in ("ffn_tc.cuh", "vad_core.cuh")]
    if not os.path.isfile(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        inc = os.path.join(os.path.dirname(os.path.dirname(os.path.realpath(nvcc))), "include")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I", inc, "-o", so, src])
    lib = C.CDLL(so)
    lib.emul_ffn_blob_bytes.restype = C.c_int
    lib.emul_ffn_pack.restype = C.c_int
    _SHIM.append(lib)
    return lib


def pack(w):
    """What a handle builds from ``w``: dict(ok, pre, post, postp, c (c1, c2, c3), blob16 uint16, blob32 float32)."""
    lib = shim()
    flat = flat_weights(w)
    scales = np.zeros(12, np.float32)
    cb = np.zeros(64 + 32 + 16, np.float32)
    b16 = np.zeros(lib.emul_ffn_blob_bytes(1) // 2, np.uint16)
    b32 = np.zeros(lib.emul_ffn_blob_bytes(0) // 4, np.float32)
    ok = lib.emul_ffn_pack(*[a.ctypes.data_as(C.c_void_p) for a in (flat, scales, cb, b16, b32)])
    return dict(ok=bool(ok), pre=scales[0:4], post=scales[4:8], postp=scales[8:12],
                c=(cb[:64], cb[64:96], cb[96:112]), blob16=b16, blob32=b32)


# ---- the bound -------------------------------------------------------------------------------------------------------
def forward64(x, w):
    """float64 forward pass: (pre-activations z_1..z_4, inputs h_0..h_3)."""
    h = np.asarray(x, np.float32).astype(np.float64)
    zs, hs = [], []
    for l in range(4):
        W = np.asarray(w["W%d" % (l + 1)], np.float32).astype(np.float64)
        b = np.asarray(w["b%d" % (l + 1)], np.float32).astype(np.float64)
        hs.append(h)
        z = h @ W + b
        zs.append(z)
        h = np.maximum(z, 0.0)
    return zs, hs


def relu_keep(z, e):
    """Units whose device value can differ from float64's: all but those with z <= -e (0 on both sides)."""
    return z > -e


def ffn_bound(x, w, impl, scales=None):
    """[n, 3] float64 bound on |device logit - float64 logit| of ``impl`` (one of IMPLS) on float32 rows ``x``.
    ``scales``: tc16_scales(w), computed when None (tc16 only)."""
    if impl not in IMPLS:
        raise ValueError(impl)
    fp16 = impl == "tc16"
    if fp16:
        ok, pre, _, sw = scales if scales is not None else tc16_scales(w)
        if not ok:
            raise ValueError("weights outside the fp16 scheme's range: the handle runs tc")
    zs, hs = forward64(x, w)
    Ws = [np.asarray(w["W%d" % (l + 1)], np.float32).astype(np.float64) for l in range(4)]
    e = np.zeros_like(hs[0])
    ds, masks = [], []
    for l in range(4):
        W = np.abs(Ws[l])
        b = np.abs(np.asarray(w["b%d" % (l + 1)], np.float32).astype(np.float64))
        K = W.shape[0]
        H = np.abs(hs[l]) + e
        HW = H @ W
        if impl == "fp32":
            d = K * U / (1 - K * U) * (HW + b)
        else:
            g = 16 if fp16 else 8
            n_acc = (3 if (fp16 and l == 0) else 2) * K_PAD[l] // g
            d = 2 * U * n_acc * HW * (1 + 2.0 ** -9)               # truncating accumulation (the a_hi B_lo half below)
            d += 2 * U * (HW + b)                                  # epilogue: two roundings to nearest
            if fp16:
                d += 3 * 2.0 ** -22 * HW
                d += 2.0 ** -25 * (W.sum(axis=0) / pre[l] + H.sum(axis=1, keepdims=True) / sw[l])
            else:
                d += 2.0 ** -19 * HW
            d *= MARGIN
        ds.append(d)
        e = e @ W + d
        if l < 3:
            keep = relu_keep(zs[l], e)
            masks.append((zs[l] > e, keep & ~(zs[l] > e)))      # (surely on, either way)
            e = np.where(keep, e, 0.0)
    # Sharper than e itself: ReLU maps an error t (h^ - h) with t = 1 on a unit that is on on both sides, t = 0 on
    # one off on both, t in [0, 1] on one that may be either.  So the logit error is exactly sum_l J_l d_l with
    # J_l the product of the later layers' W and t, and |J_l| is bounded by interval arithmetic (centre, radius).
    jc = np.broadcast_to(np.eye(3), (x.shape[0], 3, 3)).copy()
    jr = np.zeros_like(jc)
    out = np.einsum("nk,nko->no", ds[3], np.abs(jc) + jr)
    for l in (2, 1, 0):
        on, either = masks[l]
        tc = on + 0.5 * either                                  # t's centre and radius per unit
        tr = 0.5 * either
        wc = np.einsum("ko,nod->nkd", Ws[l + 1], jc)             # W_{l+1} J_{l+1}
        wr = np.einsum("ko,nod->nkd", np.abs(Ws[l + 1]), jr)
        jc, jr = tc[:, :, None] * wc, tc[:, :, None] * wr + tr[:, :, None] * (np.abs(wc) + wr)
        out += np.einsum("nk,nko->no", ds[l], np.abs(jc) + jr)
    return np.minimum(out, e)


# ---- decision rules (vad_core.cuh decide) on float32 logits -----------------------------------------------------------
def decide_argmax(logits):
    l = np.asarray(logits, np.float32)
    return ((l[:, 1] > l[:, 0]) & (l[:, 1] >= l[:, 2])).astype(np.uint8)


def decide_threshold(logits, theta):
    """(labels, decidable): speech <=> 1 / s >= theta, s = 1 + exp(l0 - l1) + exp(l2 - l1) in float32; rows whose
    1 / s lies within 2^-18 (relative) of theta are left undecided (expf and the divide are not bit-reproduced)."""
    l = np.asarray(logits, np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        s = np.float32(1) + np.exp(l[:, 0] - l[:, 1]) + np.exp(l[:, 2] - l[:, 1])
        p = np.float32(1) / s
    lab = (p >= np.float32(theta)).astype(np.uint8)
    return lab, np.abs(p.astype(np.float64) - theta) > 2.0 ** -18 * theta


# ---- weight sets -----------------------------------------------------------------------------------------------------
def glorot_x3_bias():
    """glorot(1) x 3 with N(0, 0.3) biases: larger activations, deeper fp16 scales, every bias term live."""
    from oracle import ref_math as rm
    w = {k: (v * 3.0 if k.startswith("W") else v).astype(np.float32) for k, v in rm.glorot_ffn(1).items()}
    for i in range(1, 5):
        w["b%d" % i] = np.random.default_rng(i).normal(0, 0.3, w["b%d" % i].shape).astype(np.float32)
    return w


_TRAINED = []


def trained_weights():
    """A few hundred oracle Adadelta steps from glorot(0) on scaled dataset rows of the signal catalogue (the
    weights of test_gpu_signals.py's trained_weights fixture)."""
    if not _TRAINED:
        from oracle import ref_math as rm, ref_train as rt
        import _signals
        rows = [rm.dataset_features(rm.mfcc_utterance(u)) for u in _signals.catalogue().values()]
        x = np.concatenate(rm.scale_features(rows)[0])
        y = (x[:, 0] > 0).astype(np.int64) + (x[:, 14] > 0.5)
        st = rt.init_state(rm.glorot_ffn(0))
        rng = np.random.default_rng(5)
        for _ in range(300):
            idx = rng.integers(0, x.shape[0], 256)
            rt.train_on_batch(st, x[idx], y[idx])
        _TRAINED.append({k: v.astype(np.float32) for k, v in st["p"].items()})
    return _TRAINED[0]


def deep_scaled(ea_target):
    """glorot(2) with W1..W3 scaled by one factor s chosen so that tc16_pack_weights' largest activation exponent is
    ``ea_target`` (60 is the deepest the fp16 scheme accepts; 61 makes the handle keep the tf32 path).  Rows of
    MFCC-sized features then sit 2^40 and more below the rigorous activation bounds the scales come from, so the
    fp16 operands of layers 2-4 are mostly subnormal and the subnormal floors dominate the bound."""
    from oracle import ref_math as rm
    w = {k: v.astype(np.float32) for k, v in rm.glorot_ffn(2).items()}
    bound = FEAT_BOUND.copy()
    for l in range(3):
        bound = bound @ np.abs(w["W%d" % (l + 1)].astype(np.float64))     # zero biases: the layer-4 bound goes as s^3
    s = (32000.0 * 2.0 ** (ea_target - 0.5) / bound.max()) ** (1.0 / 3.0)
    for l in range(3):
        w["W%d" % (l + 1)] = (w["W%d" % (l + 1)] * np.float32(s)).astype(np.float32)
    return w


def w4_zero():
    """glorot(0) with W4 = 0: the logits are b4 whatever the rows."""
    from oracle import ref_math as rm
    w = {k: v.astype(np.float32) for k, v in rm.glorot_ffn(0).items()}
    w["W4"] = np.zeros_like(w["W4"])
    w["b4"] = np.array([0.375, 0.8125, -1.5], np.float32)
    return w


def weight_sets():
    """name -> weights, in the order the suites use them; the first three are held to the mutant margin."""
    from oracle import ref_math as rm
    return {
        "glorot0": {k: v.astype(np.float32) for k, v in rm.glorot_ffn(0).items()},
        "glorot_x3_bias": glorot_x3_bias(),
        "trained": trained_weights(),
        "deep_ea60": deep_scaled(60),
        "beyond_ea61": deep_scaled(61),
        "w4_zero": w4_zero(),
    }
