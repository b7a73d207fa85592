"""CPU: the signal catalogue of tests/_signals.py (full-scale, tonal, band-limited, LSB-level and mixed audio) through
the host build of the kernels' per-thread arithmetic (tests/emul/emul.cpp, emul_frontend.cpp for the front end)
against the float64 oracle, at the tolerances of tests/_parity.py.  These signals leave the least headroom, so a
change to vad_core.cuh's arithmetic that eats the tolerance fails here without a GPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import ref_frontend as rf, ref_math as rm

import _signals
from _parity import mfcc_close, rows_close, decisive_rows, LOGIT_ATOL, LOGIT_RTOL
from test_emulation_cpu import emul, run_utt                      # noqa: F401  (fixture)
from test_frontend_cpu import emul as emul_fe, run_fe               # noqa: F401  (fixture)

CAT = _signals.catalogue()
HAMMING = np.hamming(400)
FRONT_ENDS = [(0.97, None), (0.97, HAMMING), (0.97, HAMMING * 32768.0)]   # the last: an int16-scaled window


def check_logits(lo, la, feats, ref_logits, ref_labels):
    fin = np.isfinite(feats).all(axis=1)
    assert np.array_equal(np.isfinite(lo).all(axis=1), fin)               # NaN rows agree exactly
    assert np.all(la[~fin] == 0)
    err = np.abs(lo[fin] - ref_logits[fin])
    assert np.all(err <= LOGIT_ATOL + LOGIT_RTOL * np.abs(ref_logits[fin])), err.max()
    dec = decisive_rows(ref_logits[fin])
    assert np.array_equal(la[fin][dec], ref_labels[fin][dec])


@pytest.mark.parametrize("name", list(CAT))
@pytest.mark.parametrize("mode", ["analyser", "dataset"])
def test_catalogue_default_path(emul, name, mode):
    lib, w = emul
    pcm = CAT[name]
    mf, fe, lo, la = run_utt(lib, pcm, mode=0 if mode == "analyser" else 1)
    c, feats, ref_logits, ref_labels = rm.vad_utterance(pcm, w, mode=mode)
    assert mfcc_close(mf, c)
    if mode == "dataset":
        assert rows_close(fe, feats)
    check_logits(lo, la, feats, ref_logits, ref_labels)


@pytest.mark.parametrize("fe_idx,name", [(i, n) for i, (_, win) in enumerate(FRONT_ENDS) for n in CAT
                                          if win is None or n not in _signals.WINDOWED_FLOAT32_FLOOR])
def test_catalogue_front_end(emul_fe, fe_idx, name):
    lib, w = emul_fe
    preemph, window = FRONT_ENDS[fe_idx]
    pcm = CAT[name]
    mf, lo, la = run_fe(lib, pcm, preemph, window)
    c, feats, ref_logits, ref_labels = rf.vad_utterance(pcm, w, preemph=preemph, window=window)
    assert mfcc_close(mf, c)
    check_logits(lo, la, feats, ref_logits, ref_labels)


def float32_frontend_mfcc(pcm, preemph, window):
    """The front end restated in float32 numpy: pre-emphasis, window and a complex64 FFT, MFCC from there in float64."""
    import scipy.fft
    x = pcm.astype(np.float32)
    y = x.copy()
    y[1:] = x[1:] - np.float32(preemph) * x[:-1]
    fr = rm.split_into_frames(y).copy()
    fr[:, :400] *= np.asarray(window, dtype=np.float32)
    X = scipy.fft.fft(fr, rm.FFT_N, axis=-1)[:, :rm.FFT_N // 2] / np.float32(rm.FFT_N)
    return rm.get_mfcc_from_spec((X.real ** 2 + X.imag ** 2).astype(np.float64), rm.get_mel_filterbanks())


@pytest.mark.parametrize("name", _signals.WINDOWED_FLOAT32_FLOOR)
def test_windowed_float32_floor(name):
    """The signals the windowed front-end checks leave out are those a float32 FFT cannot hold to the MFCC tolerance,
    and the included ones are not."""
    pcm = CAT[name]
    c = rf.mfcc_utterance(pcm, preemph=0.97, window=HAMMING)
    assert not mfcc_close(float32_frontend_mfcc(pcm, 0.97, HAMMING), c)
    for other in ("clipped_noise", "tone_1k", "mixed"):
        c = rf.mfcc_utterance(CAT[other], preemph=0.97, window=HAMMING)
        assert mfcc_close(float32_frontend_mfcc(CAT[other], 0.97, HAMMING), c)


def test_catalogue_reaches_the_rails():
    """The catalogue is only worth its cost while it holds what white noise lacks."""
    x = np.concatenate(list(CAT.values())).astype(np.int64)
    assert x.min() == -32768 and x.max() == 32767
    assert np.sum(x == -32768) > 10000 and np.sum(x == 32767) > 10000
    fr = rm.split_into_frames(CAT["tone_100_hop_periodic"])
    assert np.all(fr == fr[0])                                            # sigma5 == 0 -> NaN analyser rows
    assert np.abs(CAT["lsb_square"]).max() == 1


def test_catalogue_frames_through_spec(emul):
    """Float frames cut from the catalogue, normalised to [-1, 1] and scaled beyond int16, at frame lengths 400, 399,
    320 and 512: the per-frame FFT against the oracle's spectrum."""
    lib, _ = emul
    for n in (400, 399, 320, 512):
        for scale in (1.0, 1.0 / 32768.0, 1e5 / 32768.0):
            fr = np.stack([v[1000:1000 + n] for v in CAT.values()]).astype(np.float64) * scale
            fr = fr.astype(np.float32)
            spec = np.zeros((fr.shape[0], 256), np.float32)
            assert lib.emul_spec_f32(fr.ctypes.data_as(C.c_void_p), fr.shape[0], n,
                                     spec.ctypes.data_as(C.c_void_p)) == 0
            ref = rm.get_spec_mag(fr)
            assert np.all(np.abs(spec - ref) <= 3e-6 * ref.max(axis=1, keepdims=True))
