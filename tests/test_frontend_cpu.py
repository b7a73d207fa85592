"""CPU: the opt-in front end (pre-emphasis, analysis window) and decision threshold -- oracle semantics, the
defaults reproducing the reference path exactly (oracle/ref_frontend.py against oracle/ref_math.py), the kernels' front-end load (vad_core.cuh fft_load_pcm2_fe /
fft_load_f32_fe, driven by tests/emul/emul_frontend.cpp) against the oracle, and argument checks of the C ABI."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import ref_frontend as rf, ref_math as rm
from vad_b200.synth import synth_utterance

from test_emulation_cpu import FFN_KEYS, MFCC_ATOL, MFCC_RTOL, LOGIT_ATOL, LOGIT_RTOL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL = os.path.join(ROOT, "tests", "emul")
SO = os.path.join(EMUL, "libvademul_fe.so")
HAMMING = np.hamming(400)


@pytest.fixture(scope="module")
def emul():
    deps = [os.path.join(EMUL, f) for f in ("emul_frontend.cpp", "emul.cpp")] + \
        [os.path.join(ROOT, "vad_b200", "csrc", f) for f in ("vad_core.cuh", "vad_host_tables.h", "vad_tables.h")]
    if not os.path.isfile(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO,
                               os.path.join(EMUL, "emul_frontend.cpp")])
    lib = C.CDLL(SO)
    w = rm.glorot_ffn(0)
    flat = np.concatenate([w[k].ravel() for k in FFN_KEYS]).astype(np.float32)
    assert lib.emul_init(flat.ctypes.data_as(C.c_void_p)) == 0
    return lib, w


def logit_band(ref_logits):
    """Rows whose threshold decision the logit tolerance cannot flip.  logit(p1) = l1 - logsumexp(l0, l2) moves by at
    most |d l1| + max(|d l0|, |d l2|) <= 2 eps when every logit is within eps = LOGIT_ATOL + LOGIT_RTOL max|l|;
    a row is decisive when logit(p1) is more than twice that (4 eps) from logit(theta)."""
    eps = LOGIT_ATOL + LOGIT_RTOL * np.abs(ref_logits).max(axis=1)
    lse = np.logaddexp(ref_logits[:, 0], ref_logits[:, 2])
    return ref_logits[:, 1] - lse, 4 * eps


def threshold_decisive(ref_logits, theta):
    lp, band = logit_band(ref_logits)
    return np.abs(lp - np.log(theta / (1 - theta))) > band


# ---- oracle ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["synth_1p5s", "synth_ragged", "exact_fit", "silence_dc", "tone_noise"])
def test_oracle_defaults_reproduce_reference(golden_dir, name):
    u = np.load(os.path.join(golden_dir, "utterances.npz"))
    pcm = u[name + "/pcm"]
    w = rm.glorot_ffn(0)
    c0, f0, l0, d0 = rm.vad_utterance(pcm, w)
    c1, f1, l1, d1 = rf.vad_utterance(pcm, w, preemph=0.0, window=None, threshold=None)
    for a, b in ((c0, c1), (f0, f1), (l0, l1), (d0, d1)):
        assert np.array_equal(a, b, equal_nan=True)
    assert np.array_equal(rf.decide(l0, 0.0), d0) and np.array_equal(rf.decide(l0, -1.0), d0)
    assert np.array_equal(rf.decide(l0), d0)
    assert np.array_equal(rf.mfcc_utterance(pcm, preemph=0.0, window=None), rm.mfcc_utterance(pcm))
    assert np.array_equal(rf.preemphasis(pcm, 0.0), pcm)
    fr = rm.split_into_frames(pcm)
    if fr.shape[0]:
        assert np.array_equal(rf.get_spec_mag(fr, window=None), rm.get_spec_mag(fr))
        assert np.array_equal(rf.get_mfcc(fr, rm.get_mel_filterbanks()), rm.get_mfcc(fr, rm.get_mel_filterbanks()))


def test_oracle_preemphasis_matches_loop_and_utterance_start():
    x = synth_utterance(5, 1, 3001)
    for a in (0.0, 0.5, 0.97, 1.0):
        y = rf.preemphasis(x, a)
        ref = np.empty(len(x))
        ref[0] = x[0]
        for n in range(1, len(x)):
            ref[n] = float(x[n]) - a * float(x[n - 1])
        assert np.array_equal(np.asarray(y, dtype=np.float64), ref)
    # an utterance inside a packed buffer: the sample before it is never read
    buf = synth_utterance(5, 2, 4000)
    assert np.array_equal(rf.preemphasis(buf[1000:2000], 0.97), rf.preemphasis(buf[1000:2000].copy(), 0.97))
    assert rf.preemphasis(buf[1000:2000], 0.97)[0] == buf[1000]
    # pre-emphasis runs over the utterance before framing: frame t's first sample uses the previous frame's data
    c = rf.mfcc_utterance(x, preemph=0.97)
    fr = rm.split_into_frames(rf.preemphasis(x, 0.97))
    assert np.array_equal(c, rf.get_mfcc(fr, rm.get_mel_filterbanks()))


def test_oracle_window_and_threshold():
    rng = np.random.default_rng(1)
    fr = rng.standard_normal((3, 400)).astype(np.float32)
    spec = rf.get_spec_mag(fr, window=HAMMING)
    x = fr.astype(np.float64) * HAMMING
    ref = np.abs(np.fft.fft(x, 512, axis=-1)[:, :256] / 512.0) ** 2
    assert np.allclose(spec, ref, rtol=1e-12, atol=0)
    lg = np.array([[0.0, 0.0, 0.0], [0.0, 1.0, 0.0], [2.0, 1.0, -3.0], [np.nan] * 3])
    p1 = rf.p_voiced(lg[:3])
    assert np.allclose(p1, [1 / 3.0, np.e / (np.e + 2), np.e / (np.e + np.e ** 2 + np.e ** -3)])
    assert list(rf.decide(lg, 0.3)) == [1, 1, 0, 0]
    assert list(rf.decide(lg, 0.5)) == [0, 1, 0, 0]
    assert list(rm.decide(lg)) == [0, 1, 0, 0]


# ---- kernels' per-thread arithmetic (host emulation) --------------------------------------------------
def run_fe(lib, pcm, preemph, window, thresh=0.0, mode=0):
    T = rm.n_frames(len(pcm))
    R = max(T - 5, 0)
    mf = np.zeros((T, 13), np.float32)
    lo = np.zeros((R, 3), np.float32)
    la = np.zeros(R, np.uint8)
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    win = None if window is None else np.ascontiguousarray(window, dtype=np.float32)
    assert lib.emul_utterance_fe(pcm.ctypes.data_as(C.c_void_p), C.c_longlong(len(pcm)), mode, C.c_float(preemph),
                                 win.ctypes.data_as(C.c_void_p) if win is not None else None, C.c_float(thresh),
                                 mf.ctypes.data_as(C.c_void_p), None, lo.ctypes.data_as(C.c_void_p),
                                 la.ctypes.data_as(C.c_void_p)) == 0
    return mf, lo, la


@pytest.mark.parametrize("preemph,window", [(0.97, None), (0.0, HAMMING), (0.97, HAMMING)])
def test_emulated_frontend_load_matches_oracle(emul, preemph, window):
    lib, w = emul
    pcm = synth_utterance(77, 3, 16000 * 3 + 123)      # several steps: the previous sample crosses step buffers
    mf, lo, la = run_fe(lib, pcm, preemph, window)
    c, feats, ref_logits, ref_labels = rf.vad_utterance(pcm, w, preemph=preemph, window=window)
    assert np.all(np.abs(mf - c) <= MFCC_ATOL + MFCC_RTOL * np.abs(c))
    fin = np.isfinite(feats).all(axis=1)
    assert np.all(np.abs(lo[fin] - ref_logits[fin]) <= LOGIT_ATOL + LOGIT_RTOL * np.abs(ref_logits[fin]))
    # a wrong order (window before pre-emphasis) is far outside the tolerance
    if preemph and window is not None:
        fr = rm.split_into_frames(pcm).astype(np.float64) * HAMMING
        wrong = rf.get_mfcc(rf.preemphasis(fr, preemph), rm.get_mel_filterbanks())
        assert not np.all(np.abs(mf - wrong) <= MFCC_ATOL + MFCC_RTOL * np.abs(wrong))


@pytest.mark.parametrize("theta", [0.2, 0.5, 0.8])
def test_emulated_threshold_decision(emul, theta):
    lib, w = emul
    pcm = synth_utterance(78, 1, 16000 * 4)
    mf, lo, la = run_fe(lib, pcm, 0.97, HAMMING, thresh=theta)
    _, lo0, _ = run_fe(lib, pcm, 0.97, HAMMING, thresh=0.0)
    assert np.array_equal(lo, lo0, equal_nan=True)                   # logits do not depend on theta
    _, feats, ref_logits, ref_labels = rf.vad_utterance(pcm, w, preemph=0.97, window=HAMMING, threshold=theta)
    fin = np.isfinite(feats).all(axis=1)
    assert np.all(la[~fin] == 0)
    dec = threshold_decisive(ref_logits[fin], theta)
    assert dec.mean() > 0.5
    assert np.array_equal(la[fin][dec], ref_labels[fin][dec])


def test_emulated_frames_frontend(emul):
    lib, _ = emul
    rng = np.random.default_rng(4)
    for n, window in ((400, HAMMING), (400, None), (320, None), (512, None)):
        fr = (rng.standard_normal((3, n)) * 1234.5).astype(np.float32)
        spec = np.zeros((3, 256), np.float32)
        win = None if window is None else np.ascontiguousarray(window, dtype=np.float32)
        assert lib.emul_spec_f32_fe(fr.ctypes.data_as(C.c_void_p), 3, n, C.c_float(0.97),
                                    win.ctypes.data_as(C.c_void_p) if win is not None else None,
                                    spec.ctypes.data_as(C.c_void_p)) == 0
        ref = rf.get_spec_mag(rf.preemphasis(fr, 0.97), window=window)   # each frame is its own signal
        assert np.max(np.abs(spec - ref)) <= 3e-6 * ref.max()


# ---- C ABI -------------------------------------------------------------------------------------------
def test_cabi_rejects_null_handle():
    from vad_b200 import build, _lib
    build.build()
    lib = _lib.load()
    win = np.ones(400, np.float32)
    assert lib.vadb200_set_frontend(None, 0.97, win.ctypes.data_as(C.c_void_p)) == -1
    assert lib.vadb200_get_frontend(None, None, None, None) == -1
    assert lib.vadb200_set_decision_threshold(None, 0.5) == -1
    assert np.isnan(lib.vadb200_get_decision_threshold(None))
    assert lib.vadb200_version() == 201
