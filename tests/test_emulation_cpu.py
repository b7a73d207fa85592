"""CPU: the exact per-thread fp32 arithmetic of the CUDA kernels (vad_b200/csrc/vad_core.cuh),
compiled with g++ and driven through the kernels' 16-threads-per-frame dataflow by
tests/emul/emul.cpp, against the float64 oracle.  Validates index math (FFT passes, transpose,
partner exchange, bin ownership, mel groups, ring, block phases) and accuracy with no GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import ref_math as rm
from vad_b200.synth import synth_utterance

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "emul", "emul.cpp")
SO = os.path.join(ROOT, "tests", "emul", "libvademul.so")
FFN_KEYS = ["W1", "b1", "W2", "b2", "W3", "b3", "W4", "b4"]

MFCC_ATOL, MFCC_RTOL = 1e-4, 1e-4       # north_star / SURVEY 8(d)
LOGIT_ATOL, LOGIT_RTOL = 1e-3, 1e-3


@pytest.fixture(scope="module")
def emul():
    deps = [SRC] + [os.path.join(ROOT, "vad_b200", "csrc", f) for f in
                    ("vad_core.cuh", "vad_host_tables.h", "vad_tables.h")]
    if not os.path.isfile(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-x", "c++", "-o", SO, SRC])
    lib = C.CDLL(SO)
    w = rm.glorot_ffn(0)
    flat = np.concatenate([w[k].ravel() for k in FFN_KEYS]).astype(np.float32)
    assert lib.emul_init(flat.ctypes.data_as(C.c_void_p)) == 0
    return lib, w


def run_utt(lib, pcm, mode=0):
    T = rm.n_frames(len(pcm))
    R = max(T - 5, 0)
    mf = np.zeros((T, 13), np.float32)
    fe = np.zeros((R, 39), np.float32)
    lo = np.zeros((R, 3), np.float32)
    la = np.zeros(R, np.uint8)
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    assert lib.emul_utterance(pcm.ctypes.data_as(C.c_void_p), C.c_longlong(len(pcm)), mode,
                              mf.ctypes.data_as(C.c_void_p), fe.ctypes.data_as(C.c_void_p),
                              lo.ctypes.data_as(C.c_void_p), la.ctypes.data_as(C.c_void_p)) == 0
    return mf, fe, lo, la


def check_against_oracle(lib, w, pcm):
    mf, fe, lo, la = run_utt(lib, pcm)
    c, feats, logits, labels = rm.vad_utterance(pcm, w)
    assert np.all(np.abs(mf - c) <= MFCC_ATOL + MFCC_RTOL * np.abs(c))
    if feats.shape[0] == 0:
        return
    fin = np.isfinite(feats).all(axis=1)
    assert np.array_equal(np.isfinite(lo).all(axis=1), fin)            # nan rows agree
    assert np.all(la[~fin] == 0)
    err = np.abs(lo[fin] - logits[fin])
    assert np.all(err <= LOGIT_ATOL + LOGIT_RTOL * np.abs(logits[fin]))
    srt = np.sort(logits[fin], axis=1)
    decisive = (srt[:, -1] - srt[:, -2]) > 2 * (LOGIT_ATOL + LOGIT_RTOL * np.abs(srt[:, -1]))
    assert np.array_equal(la[fin][decisive], labels[fin][decisive])


def test_spectrum_kat(emul, golden_dir):
    lib, _ = emul
    kat = np.load(os.path.join(golden_dir, "kat_frame.npz"))
    fr = kat["frame"].astype(np.float32)[None].copy()
    spec = np.zeros((1, 256), np.float32)
    lib.emul_spec_f32(fr.ctypes.data_as(C.c_void_p), 1, 400, spec.ctypes.data_as(C.c_void_p))
    ref = rm.get_spec_mag(kat["frame"])
    assert np.max(np.abs(spec[0] - ref)) <= 2e-6 * ref.max()


@pytest.mark.parametrize("name", ["synth_1p5s", "synth_ragged", "exact_fit", "silence_dc", "tone_noise"])
def test_golden_utterances(emul, golden_dir, name):
    lib, w = emul
    u = np.load(os.path.join(golden_dir, "utterances.npz"))
    pcm = u[name + "/pcm"]
    check_against_oracle(lib, w, pcm)
    mf, fe, lo, la = run_utt(lib, pcm)
    # straight against the frozen reference outputs as well
    assert np.all(np.abs(mf - u[name + "/mfcc"]) <= MFCC_ATOL + MFCC_RTOL * np.abs(u[name + "/mfcc"]))
    ds = run_utt(lib, pcm, mode=1)[1]
    ref_ds = u[name + "/dataset_rows"]
    assert np.all(np.abs(ds - ref_ds) <= 3e-4 + 1e-4 * np.abs(ref_ds))


def test_long_utterance_ring_wrap(emul):
    lib, w = emul
    check_against_oracle(lib, w, synth_utterance(77, 1, 16000 * 12 + 123))   # > 4 block phases, ring wraps


def test_full_scale_and_tiny_amplitudes(emul):
    lib, w = emul
    rng = np.random.default_rng(3)
    loud = np.clip(rng.standard_normal(8000) * 20000, -32768, 32767).astype(np.int16)
    quiet = (rng.integers(-2, 3, 8000)).astype(np.int16)
    square = (np.where((np.arange(8000) // 37) % 2 == 0, 32767, -32768)).astype(np.int16)
    for pcm in (loud, quiet, square):
        mf, _, _, _ = run_utt(lib, pcm)
        c = rm.mfcc_utterance(pcm)
        assert np.all(np.abs(mf - c) <= MFCC_ATOL + MFCC_RTOL * np.abs(c))
