"""CPU: what tests/_mfcc_bound.py's spectrum -> MFCC bound and tests/_window_bound.py's window-feature rules catch.

* The FFT's precision, which the GPU suite does not bound (it holds the device to the bit-exact replay): the replayed
  float32 |2X|^2 stays within a small fraction of fft_bound's componentwise bound, and mutants of the replay --
  twiddles with 11 significant bits, one W512 conjugated, one bin pair swapped -- exceed it.
* Faithful emulations stay inside the bounds: the replay's own MFCC rows (vad_core.cuh's mel2_run / dct_coef2 through
  tests/emul), numpy float32 mel / log2 / DCT in the kernels' chain orders and reversed within the chains, and the
  window arithmetic over replayed MFCC rows.
* Mutants fail by at least MUTANT_FACTOR on the catalogue: a triangle's last bin dropped, the mel scale 2^-19, log2
  to about 12 bits, the folded DCT in fp16 or tf32, lifter indices shifted by one; the mean over four frames, sigma
  with ddof = 1, a one-pass float32 variance, the analyser d2 from c2 instead of z.

Each test prints the fraction of the bound used or the factor by which a mutant fails."""
import ctypes as C

import numpy as np

from oracle import ref_math as rm

import _mfcc_bound as mb
import _signals
import _window_bound as wb

MUTANT_FACTOR = 5.0
CAT = _signals.catalogue()
F32 = np.float32


def utt_mfcc_feats(pcm, mode):
    """The replay's MFCC rows [T, 13] and feature rows [T - 5, 39] (tests/emul/emul.cpp emul_utterance)."""
    lib = mb.shim()
    T = rm.n_frames(len(pcm))
    mf = np.zeros((T, 13), np.float32)
    fe = np.zeros((max(T - 5, 0), 39), np.float32)
    pcm = np.ascontiguousarray(pcm, np.int16)
    assert lib.emul_utterance(pcm.ctypes.data_as(C.c_void_p), C.c_longlong(len(pcm)), mode,
                              mf.ctypes.data_as(C.c_void_p), fe.ctypes.data_as(C.c_void_p), None, None) == 0
    return mf, fe


# ---- the replay's FFT against the componentwise bound ----------------------------------------------------------------
def frames_of(name):
    return rm.split_into_frames(CAT[name]).astype(np.float32)


FFT_SIGNALS = ("clipped_noise", "tone_1k", "chirp_50_8k", "lsb_noise", "mixed")


def fft_fraction(P32, P64, bound, lo=mb.MEL_FIRST_BIN):
    d = np.abs(np.asarray(P32, np.float64)[:, lo:] - P64[:, lo:])
    return float(np.max(d / bound[:, lo:]))


def test_replayed_spectrum_within_fft_bound():
    worst = 0.0
    for name in FFT_SIGNALS:
        fr = frames_of(name)
        P64, bnd = mb.fft_bound(fr)
        worst = max(worst, fft_fraction(mb.power_f32(fr), P64, bnd, 0))
        # the fused kernel's PCM load (fft_load_pcm2, NZ = 13) gives the same bits as the float-frame load
        assert np.array_equal(mb.power_pcm(CAT[name])[:, 10:], mb.power_f32(fr)[:, 10:])
    print("\nreplayed |2X|^2: worst |d| / fft_bound = %.4f" % worst)
    assert worst < 0.05


def round_sig(x, bits):
    m, e = np.frexp(np.asarray(x, np.float64))
    return (np.round(m * 2.0 ** bits) / 2.0 ** bits * 2.0 ** e).astype(np.float32)


def test_fft_mutants_exceed_bound():
    tw1, tw2 = mb.twiddles()
    mutants = {"twiddles_11_bits": (round_sig(tw1, 11), round_sig(tw2, 11), None),
               "one_w512_conjugated": (tw1, tw2 * np.where(np.arange(128)[:, None] == 37, [1, -1], [1, 1]), None),
               "bin_pair_swapped": (tw1, tw2, (60, 61))}
    out = {}
    try:
        for mname, (t1, t2, swap) in mutants.items():
            mb.twiddles((t1, t2))
            worst = []
            for name in FFT_SIGNALS:
                fr = frames_of(name)
                P = mb.power_f32(fr)
                if swap:
                    P[:, list(swap)] = P[:, list(swap[::-1])]
                P64, bnd = mb.fft_bound(fr)
                worst.append(fft_fraction(P, P64, bnd))
            out[mname] = worst
    finally:
        mb.twiddles((tw1, tw2))
    print("\nFFT mutants, |d| / fft_bound per signal %s:" % (FFT_SIGNALS,))
    for k, v in out.items():
        print("  %-22s %s" % (k, " ".join("%9.1f" % f for f in v)))
        assert max(v) >= MUTANT_FACTOR, k
    assert min(out["twiddles_11_bits"]) >= MUTANT_FACTOR


# ---- MFCC stages -----------------------------------------------------------------------------------------------------
def test_tables_of_both_mel_and_dct_paths_agree():
    t = mb.tables()
    assert np.array_equal(t["melw"], t["melw2"]) and np.array_equal(t["dct"], t["dctp"])
    fb = mb.filterbank()
    assert np.array_equal(t["melw"] != 0, fb != 0)
    assert np.max(np.abs(t["melw"] - fb * 2.0 ** -20) / np.where(fb > 0, fb * 2.0 ** -20, 1)) <= 2.0 ** -24
    assert np.max(np.abs(t["dct"] - mb.dct64())) <= 2.0 ** -24 * np.abs(mb.dct64()).max()


CHAINS = [list(range(j, 26, 4)) for j in range(4)]


def emul_mel(P, w, reverse=False):
    """mel2_run per frame: for filter m, two FFMA chains over pair rows (parity of the pair index), each frame lane
    the even / odd bins of a pair; lanes' chains merged, then the two bins' sums added.  float32 throughout."""
    P = np.asarray(P, np.float32)
    out = np.zeros((P.shape[0], 26), np.float32)
    for m in range(26):
        nz = np.flatnonzero(w[m])
        q0, q1 = nz[0] // 2, nz[-1] // 2 + 1
        acc = np.zeros((2, 2, P.shape[0]), np.float32)          # [chain i & 1][bin e]
        qs = list(range(q0, q1))
        for i, q in (reversed(list(enumerate(qs))) if reverse else enumerate(qs)):
            for e in range(2):
                b = 2 * q + e
                acc[i & 1, e] = (P[:, b].astype(np.float64) * w[m, b] + acc[i & 1, e]).astype(np.float32)
        s = acc[0] + acc[1]
        out[:, m] = s[0] + s[1]
    return out


def emul_log2(E, bits=None):
    L = np.log2(np.where(E == 0, F32(rm.EPS), E)).astype(np.float32)
    return L if bits is None else round_sig(L, bits)


def emul_dct(L, D, reverse=False):
    """dct_coef's four FFMA chains (n % 4), merged (a0 + a2) + (a1 + a3); reverse: each chain from its last term."""
    L = np.asarray(L, np.float32)
    out = np.zeros((L.shape[0], D.shape[0]), np.float32)
    for k in range(D.shape[0]):
        a = []
        for ch in CHAINS:
            acc = np.zeros(L.shape[0], np.float32)
            for n in (ch[::-1] if reverse else ch):
                acc = (L[:, n].astype(np.float64) * float(D[k, n]) + acc).astype(np.float32)
            a.append(acc)
        out[:, k] = (a[0] + a[2]) + (a[1] + a[3])
    return out


def fraction(C, ref, bnd):
    d = np.abs(np.asarray(C, np.float64) - ref)
    return float(np.max(d / bnd))


def test_faithful_mfcc_within_bound():
    t = mb.tables()
    worst = {}
    for name, pcm in CAT.items():
        P = mb.power_pcm(pcm)
        ref, bnd, _ = mb.mfcc_bound(P)
        mf, _ = utt_mfcc_feats(pcm, 0)
        cases = {"replay (mel2_run, dct_coef2)": mf}
        for rev in (False, True):
            E = emul_mel(np.nan_to_num(P), t["melw2"], rev)
            cases["numpy %s" % ("reversed" if rev else "kernel order")] = emul_dct(emul_log2(E), t["dct"], rev)
        for k, C_ in cases.items():
            f = fraction(C_, ref, bnd)
            assert f <= 1.0, (name, k, f)
            worst[k] = max(worst.get(k, 0.0), f)
    print("\nfaithful MFCC, worst |d| / bound:")
    for k, v in worst.items():
        print("  %-30s %.4f" % (k, v))
    assert max(worst.values()) < 0.5


def lifter_shifted(D):
    lf = rm.lifter_coefs(14)
    return (D.astype(np.float64) / lf[:13, None] * lf[1:14, None]).astype(np.float32)


def tf32(a):
    return (np.asarray(a, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def last_bin_dropped(w):
    w = w.copy()
    for m in range(26):
        w[m, np.flatnonzero(w[m])[-1]] = 0
    return w


MFCC_MUTANTS = {
    "last_triangle_bin_dropped": lambda P, t: emul_dct(emul_log2(emul_mel(P, last_bin_dropped(t["melw2"]))), t["dct"]),
    "mel_scale_2^-19": lambda P, t: emul_dct(emul_log2(emul_mel(P, t["melw2"] * F32(2))), t["dct"]),
    "log2_12_bits": lambda P, t: emul_dct(emul_log2(emul_mel(P, t["melw2"]), bits=12), t["dct"]),
    "dct_fp16": lambda P, t: emul_dct(emul_log2(emul_mel(P, t["melw2"])), t["dct"].astype(np.float16).astype(F32)),
    "dct_tf32": lambda P, t: emul_dct(emul_log2(emul_mel(P, t["melw2"])), tf32(t["dct"])),
    "lifter_shifted": lambda P, t: emul_dct(emul_log2(emul_mel(P, t["melw2"])), lifter_shifted(t["dct"])),
}


def test_mfcc_mutants_exceed_bound():
    t = mb.tables()
    res = {k: {} for k in MFCC_MUTANTS}
    for name, pcm in CAT.items():
        P = np.nan_to_num(mb.power_pcm(pcm))
        ref, bnd, _ = mb.mfcc_bound(P)
        for k, f in MFCC_MUTANTS.items():
            res[k][name] = fraction(f(P, t), ref, bnd)
    print("\nMFCC mutants, worst |d| / bound (lowest signal):")
    for k, v in res.items():
        lo = min(v, key=v.get)
        print("  %-28s %10.1f   lowest %8.1f on %s" % (k, max(v.values()), v[lo], lo))
        # every mutant fails on every catalogue signal except where noted
        assert max(v.values()) >= MUTANT_FACTOR, k
    # the mel scale moves every log-energy by exactly 1 (the DCT rows k >= 1 sum to ~0): it shows on c0 of every signal
    for k in res:
        assert min(res[k].values()) >= MUTANT_FACTOR, (k, res[k])


# ---- window features -------------------------------------------------------------------------------------------------
def test_replayed_window_features_follow_the_rules():
    worst = {}
    for name, pcm in CAT.items():
        for mode, mname in ((0, "analyser"), (1, "dataset")):
            mf, fe = utt_mfcc_feats(pcm, mode)
            r = wb.window_check(mf, fe, mname, "scalar")
            for k, v in r.items():
                worst[k] = max(worst.get(k, 0.0), v)
    print("\nreplayed window features, worst |d| / bound: %s" % worst)
    assert max(worst.values()) < 0.75


def emul_window(w, variant=None):
    """[n, 5, 13] float32 windows -> (z, d2) in float32, the packed arithmetic of window_features_pairs or a mutant."""
    c = [np.asarray(w[:, d], np.float32) for d in range(5)]
    if variant == "mean_of_four":
        mu = (((c[0] + c[1]) + c[2]) + c[3]) * F32(0.25)
    else:
        mu = ((((c[0] + c[1]) + c[2]) + c[3]) + c[4]) * F32(0.2)
    d = [ci - mu for ci in c]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        if variant == "one_pass_variance":
            sq = c[0] * c[0]
            for ci in c[1:]:
                sq = (ci.astype(np.float64) * ci + sq).astype(np.float32)
            var = sq * F32(0.2) - mu * mu
        else:
            q = d[0] * d[0]
            for di in d[1:]:
                q = (di.astype(np.float64) * di + q).astype(np.float32)
            var = q * (F32(0.25) if variant == "ddof_1" else F32(0.2))
        z = d[2] * (F32(1) / np.sqrt(var))
        zz = c[2] if variant == "d2_from_c2" else z
        d2 = (c[4] - zz) - (zz - c[0])
    return z, d2


def test_window_mutants_exceed_bound():
    res = {}
    for name, pcm in CAT.items():
        mf, _ = utt_mfcc_feats(pcm, 0)
        w = wb.windows(mf)
        zr, zb, dr, db = wb.analyser_bound(w)
        ok = ~wb.nan_rule(w, "pairs")
        for variant in (None, "mean_of_four", "ddof_1", "one_pass_variance", "d2_from_c2"):
            z, d2 = emul_window(w, variant)
            with np.errstate(invalid="ignore", divide="ignore"):
                f = max(np.nanmax(np.where(ok, np.abs(z - zr) / zb, 0)), np.nanmax(np.where(ok, np.abs(d2 - dr) / db, 0)))
                if not np.isfinite(z[ok]).all() or not np.isfinite(d2[ok]).all():
                    f = np.inf
            res.setdefault(variant, {})[name] = f
    print("\nwindow mutants, worst |d| / bound (lowest signal):")
    for k, v in res.items():
        lo = min(v, key=v.get)
        print("  %-20s %10.1f   lowest %8.3g on %s" % (k or "faithful (packed)", max(v.values()), v[lo], lo))
    assert max(res[None].values()) < 0.75
    for k in ("mean_of_four", "ddof_1", "one_pass_variance", "d2_from_c2"):
        assert max(res[k].values()) >= MUTANT_FACTOR, k
