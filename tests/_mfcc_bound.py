"""Per-entry rounding bound of the MFCC rows on the kernel's own float32 power spectrum (tests/ only).

The chain is split at the power spectrum.  The FFT is vad_core.cuh's __host__ __device__ code: on the device every
operation is rounded explicitly (__fadd2_rn, __ffma2_rn, fmaf) and the twiddles are the host's own tables, so the g++
build of the same code in tests/emul/emul_frontend.cpp (compiled with -ffp-contract=off) reproduces the device's
float32 |2X|^2 bit for bit; ``power_pcm`` / ``power_f32`` return it.  A componentwise bound through the 512-point FFT
is far looser than the real error (it sums every input path's rounding), so the FFT is held to that replay instead,
and its own precision is checked on the CPU against ``fft_bound``.

``mfcc_bound(P)`` takes float32 powers P = |2X|^2 and returns the float64 reference MFCC of the reference's semantics
(oracle/ref_math.py get_mfcc_from_spec on P 2^-20: float64 filterbank, == 0 -> eps, log10, DCT-II ortho, lifter 22)
and a bound on |device - reference| per entry, for any device that evaluates, with u = 2^-24 and
gamma_n = n u / (1 - n u):

* mel: E_m = sum_k w_mk P_k with the stored float32 weights w (x 2^-20, exact scale) as FFMA chains in any order and
  any split into chains: the terms are non-negative, so the rounding is within gamma_n sum_k w_mk P_k with n the
  filter's bins (+ 4 for the chain merges), plus n 2^-149 should partial sums be subnormal.  The weights' deviation
  from the float64 filterbank is taken exactly from the stored values: sum_k |w_mk - fb_mk 2^-20| P_k.
* log2: __log2f errs by at most 2^-22 absolutely for E in [0.5, 2] and by 2 ulp of the result elsewhere (CUDA C++
  Programming Guide, intrinsic functions); the mel error dE passes on as -log2(1 - dE / E).  E == 0 takes the eps
  branch (log2 = -52) only when every contributing bin is exactly 0, on both sides (asserted).  Every non-zero E must be a normal float32 (asserted): MUFU.LG2 flushes subnormals.
* DCT: C_k = sum_n D_kn L_n with the folded float32 coefficients D (lifter x DCT-II x log10 2).  dct_coef,
  dct_coef2 and dct_coef4 run the same four FFMA chains (at most 7 long) and merge them in a two-level tree, so
  gamma_9 sum_n |D_kn| |L_n| covers all three in any order within the chains (gamma_28, which would also cover one
  26-long chain, is three times looser and above the flat tolerance for most of c6..c12); the coefficients'
  deviation from float64 (lifter and log10 2 included) is taken exactly; the log error passes on through |D|.

Everything is first order in u; MARGIN covers the second-order terms."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import ref_math as rm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL = os.path.join(ROOT, "tests", "emul")
SO = os.path.join(EMUL, "libvademul_fe.so")
U = 2.0 ** -24
MARGIN = 1.0 + 2.0 ** -9
LOG2_ABS = 2.0 ** -22
MEL_FIRST_BIN = 10
EPS = rm.EPS


# The DCT's chains: log-energy n goes to chain n % 4 (7, 7, 6, 6 FFMAs), merged as (a0 + a2) + (a1 + a3) --
# dct_coef, and per coefficient dct_coef2 / dct_coef4 (bit-identical chains).  No product passes through more than
# 7 + 2 roundings, in whatever order each chain runs.
DCT_DEPTH = 9


def gamma(n):
    return n * U / (1 - n * U)


def ulp32(x):
    """float32 ulp of |x| (x normal)."""
    return 2.0 ** (np.floor(np.log2(np.maximum(np.abs(x), 2.0 ** -126))) - 23)


# ---- the host replay (tests/emul/emul_frontend.cpp) ------------------------------------------------------------------
_LIB = []


def shim():
    if _LIB:
        return _LIB[0]
    deps = [os.path.join(EMUL, f) for f in ("emul_frontend.cpp", "emul.cpp")] + \
        [os.path.join(ROOT, "vad_b200", "csrc", f) for f in ("vad_core.cuh", "vad_host_tables.h", "vad_tables.h")]
    if not os.path.isfile(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO,
                               os.path.join(EMUL, "emul_frontend.cpp")])
    lib = C.CDLL(SO)
    assert lib.emul_init(None) == 0
    _LIB.append(lib)
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _fe_args(fe):
    """fe: None (no front end) or (preemph, window: 400 weights or None)."""
    if fe is None:
        return 0, C.c_float(0.0), None
    win = None if fe[1] is None else np.ascontiguousarray(fe[1], np.float32)
    return 1, C.c_float(fe[0]), win


def power_pcm(pcm, fe=None):
    """[T, 256] float32 |2X|^2 of every frame of one utterance through the fused kernel's load path; bins below
    MEL_FIRST_BIN (which the kernel drops) are NaN."""
    pcm = np.ascontiguousarray(pcm, np.int16)
    out = np.full((rm.n_frames(len(pcm)), 256), np.nan, np.float32)
    use, a, win = _fe_args(fe)
    assert shim().emul_power_pcm(_ptr(pcm), C.c_longlong(len(pcm)), use, a, _ptr(win), _ptr(out)) == 0
    return out


def power_f32(frames, fe=None):
    """[n, 256] float32 |2X|^2 of explicit float32 frames [n, frame_len] through frames_kernel's load path."""
    fr = np.ascontiguousarray(frames, np.float32)
    out = np.full((fr.shape[0], 256), np.nan, np.float32)
    use, a, win = _fe_args(fe)
    assert shim().emul_power_f32(_ptr(fr), fr.shape[0], fr.shape[1], use, a, _ptr(win), _ptr(out)) == 0
    return out


def spec_f32(frames, fe=None):
    """get_spec_mag as frames_kernel computes it: |2X|^2 x 2^-20 in float32."""
    return power_f32(frames, fe) * np.float32(2.0 ** -20)


def twiddles(tw=None):
    """(tw1 [256, 2], tw2 [128, 2]) the replay uses; with ``tw`` given, replace them (emul reinit restores)."""
    lib = shim()
    if tw is None:
        t1, t2 = np.zeros((256, 2), np.float32), np.zeros((128, 2), np.float32)
        assert lib.emul_twiddles(_ptr(t1), _ptr(t2), 0) == 0
        return t1, t2
    t1, t2 = (np.ascontiguousarray(t, np.float32) for t in tw)
    assert lib.emul_twiddles(_ptr(t1), _ptr(t2), 1) == 0


_TABLES = {}


def tables():
    """The float32 tables the kernels read: melw, melw2 [26, 256] (x 2^-20), dct, dctp [13, 26]."""
    if not _TABLES:
        t = {k: np.zeros((26, 256), np.float32) for k in ("melw", "melw2")}
        t.update({k: np.zeros((13, 26), np.float32) for k in ("dct", "dctp")})
        assert shim().emul_tables(*[_ptr(t[k]) for k in ("melw", "melw2", "dct", "dctp")]) == 0
        _TABLES.update(t)
    return _TABLES


def filterbank():
    return rm.get_mel_filterbanks()


def dct64():
    """float64 lifter x DCT-II ortho x log10(2): the reference's log10 / DCT / lifter applied to log2 energies."""
    return rm.dct2_ortho_matrix(13, 26) * rm.lifter_coefs(13)[:, None] * np.log10(2.0)


# ---- the bound -------------------------------------------------------------------------------------------------------
def mfcc_bound(P, melw=None, dct=None):
    """(ref [n, 13], bound [n, 13], stages) for float32 powers P [n, 256] (bins below MEL_FIRST_BIN ignored).
    melw / dct: the float32 tables (default: the kernels' own; the CPU suite passes mutated ones).  stages holds
    the float64 mel energies E, their bound dE, log2 energies L and their bound dL."""
    P = np.asarray(P, np.float32).astype(np.float64)[:, MEL_FIRST_BIN:]
    fb = filterbank()
    assert not fb[:, :MEL_FIRST_BIN].any()
    fb = fb[:, MEL_FIRST_BIN:]
    w = (tables()["melw"] if melw is None else np.asarray(melw, np.float32)).astype(np.float64)[:, MEL_FIRST_BIN:]
    D = (tables()["dct"] if dct is None else np.asarray(dct, np.float32)).astype(np.float64)
    assert np.isfinite(P).all() and (P >= 0).all()
    support = fb != 0
    # mel
    E = (P @ fb.T) * 2.0 ** -20
    Sw = P @ w.T
    n = support.sum(axis=1) + 4
    dE = gamma(n) * Sw + n * 2.0 ** -149 + P @ np.abs(w - fb * 2.0 ** -20).T
    zero = E == 0
    assert np.array_equal(zero, (P @ support.T) == 0), "eps branch where a contributing bin is not zero"
    # log2
    with np.errstate(divide="ignore", invalid="ignore"):
        rel = np.where(zero, 0.0, dE / np.where(zero, 1.0, E))
        assert np.all(zero | (E * (1 - rel) >= 2.0 ** -126)), "a mel energy may be subnormal"
        L = np.where(zero, np.log2(EPS), np.log2(np.where(zero, 1.0, E)))
        dL = np.where(rel < 1, -np.log2(1 - np.minimum(rel, 0.5)), np.inf)
    dL = dL + np.where((E * (1 - rel) >= 0.5) & (E * (1 + rel) <= 2.0), LOG2_ABS, 2 * ulp32(np.abs(L) + dL))
    # DCT
    D64 = dct64()
    La = np.abs(L) + dL
    dC = gamma(DCT_DEPTH) * (La @ np.abs(D).T) + La @ np.abs(D - D64).T + dL @ np.abs(D64).T
    dC += 2.0 ** -40 * (La @ np.abs(D64).T)          # the oracle's own float64 rounding
    P0 = np.zeros((P.shape[0], 256))
    P0[:, MEL_FIRST_BIN:] = P
    ref = rm.get_mfcc_from_spec(P0 * 2.0 ** -20, filterbank())
    return ref, dC * MARGIN, dict(E=E, dE=dE, L=L, dL=dL)


# ---- componentwise FFT bound (CPU suite only) ------------------------------------------------------------------------
FFT_STAGE = 4 * U      # per radix-2 butterfly output component: o0 two FFMAs, o1 = 2a - o0 one more, the W16 constant


def _bfly(a, ra, b, rb, w):
    """a + w b, a - w b with radii: (v0, r0, v1, r1); a, b complex [..], ra / rb (re, im) radius pairs."""
    wb = w * b
    wr, wi = abs(w.real), abs(w.imag)
    rwb = (wr * rb[0] + wi * rb[1], wr * rb[1] + wi * rb[0])
    mag = (np.abs(a.real) + wr * np.abs(b.real) + wi * np.abs(b.imag) + ra[0] + rwb[0],
           np.abs(a.imag) + wr * np.abs(b.imag) + wi * np.abs(b.real) + ra[1] + rwb[1])
    r = (ra[0] + rwb[0] + FFT_STAGE * mag[0], ra[1] + rwb[1] + FFT_STAGE * mag[1])
    return a + wb, r, a - wb, r


def _dft16(v, r):
    """Radix-2 decimation in time over the last axis (16), natural order in and out, with radii."""
    rev = [int("{:04b}".format(i)[::-1], 2) for i in range(16)]
    v = v[..., rev]
    r = (r[0][..., rev], r[1][..., rev])
    m = 1
    while m < 16:
        v2, r2 = v.copy(), (r[0].copy(), r[1].copy())
        for start in range(0, 16, 2 * m):
            for k in range(m):
                i, j = start + k, start + k + m
                w = np.exp(-2j * np.pi * k / (2 * m))
                o0, q0, o1, q1 = _bfly(v[..., i], (r[0][..., i], r[1][..., i]), v[..., j],
                                       (r[0][..., j], r[1][..., j]), w)
                v2[..., i], v2[..., j] = o0, o1
                r2[0][..., i], r2[1][..., i], r2[0][..., j], r2[1][..., j] = q0[0], q0[1], q1[0], q1[1]
        v, r, m = v2, r2, 2 * m
    return v, r


def fft_bound(frames):
    """(P64 [n, 256] exact |2X|^2 of float32 frames (<= 512 samples, no front end), bound [n, 256]): a componentwise
    bound on the float32 |2X|^2 of vad_core.cuh's FFT, written out per radix-2 stage of dft16 (FFT_STAGE per output
    component), per inter-pass twiddle (two roundings and the table's own rounding) and per real-FFT split (two
    FFMAs for 2X, one more for the mirror bin, then |.|^2 as FFMA + FMUL).  Loose by construction: it sums every
    path's rounding (an l1 sum) where the real error grows like an l2 sum."""
    fr = np.asarray(frames, np.float32).astype(np.float64)
    x = np.zeros((fr.shape[0], 512))
    x[:, :fr.shape[1]] = fr
    z = x[:, 0::2] + 1j * x[:, 1::2]                          # [n, 256]
    zero = np.zeros(z.shape)
    # pass 1: thread t, DFT16 over j of z[t + 16 j]
    v = z.reshape(-1, 16, 16).transpose(0, 2, 1)               # [n, t, j]
    v, r = _dft16(v, (zero.reshape(-1, 16, 16), zero.reshape(-1, 16, 16)))
    t = np.arange(16)[:, None]
    k1 = np.arange(16)[None, :]
    w = np.exp(-2j * np.pi * t * k1 / 256.0)                   # [t, k1]
    wr, wi = np.abs(w.real), np.abs(w.imag)
    wv = w * v
    mag = (wr * np.abs(v.real) + wi * np.abs(v.imag) + wr * r[0] + wi * r[1],
           wr * np.abs(v.imag) + wi * np.abs(v.real) + wr * r[1] + wi * r[0])
    r = (wr * r[0] + wi * r[1] + 3 * U * mag[0], wr * r[1] + wi * r[0] + 3 * U * mag[1])
    v = wv
    # pass 2: thread k1, DFT16 over t -> Z[k1 + 16 k2]
    v, r = _dft16(v.transpose(0, 2, 1), (r[0].transpose(0, 2, 1), r[1].transpose(0, 2, 1)))
    Z = v.transpose(0, 2, 1).reshape(-1, 256)                  # index k2 * 16 + k1 after the transpose
    Zr = (r[0].transpose(0, 2, 1).reshape(-1, 256), r[1].transpose(0, 2, 1).reshape(-1, 256))
    k = np.arange(256)
    a, ra = Z[:, k], (Zr[0][:, k], Zr[1][:, k])
    m = (256 - k) % 256
    b, rb = np.conj(Z[:, m]), (Zr[0][:, m], Zr[1][:, m])
    Ev, Er = a + b, (ra[0] + rb[0] + U * (np.abs((a + b).real) + ra[0] + rb[0]),
                     ra[1] + rb[1] + U * (np.abs((a + b).imag) + ra[1] + rb[1]))
    Ov = -1j * (a - b)
    Or = (ra[1] + rb[1] + U * (np.abs(Ov.real) + ra[1] + rb[1]), ra[0] + rb[0] + U * (np.abs(Ov.imag) + ra[0] + rb[0]))
    w5 = np.exp(-2j * np.pi * k / 512.0)
    X, Xr, _, _ = _bfly(Ev, Er, Ov, Or, w5)                    # 2X[k] = E + w O (the mirror bin's 2E - X: same radius)
    Xr = (Xr[0] + U * np.abs(w5.real) * np.abs(Ov.real), Xr[1] + U * np.abs(w5.imag) * np.abs(Ov.imag))
    Xr = (Xr[0] + 2 * U * (np.abs(X.real) + Xr[0]), Xr[1] + 2 * U * (np.abs(X.imag) + Xr[1]))   # mirror: one more
    P = np.abs(X) ** 2
    ax, ay = np.abs(X.real) + Xr[0], np.abs(X.imag) + Xr[1]
    dP = 2 * np.abs(X.real) * Xr[0] + Xr[0] ** 2 + 2 * np.abs(X.imag) * Xr[1] + Xr[1] ** 2 + 2 * U * (ax * ax + ay * ay)
    return P, dP * MARGIN
