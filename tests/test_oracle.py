"""CPU: pin the oracle restatement (oracle/ref_math.py, oracle/ref_loop.py, oracle/ref_io.py) against
the golden vectors frozen from the unmodified reference (oracle/make_golden.py)."""
import os

import numpy as np
import pytest

from oracle import ref_math as rm, ref_loop


@pytest.fixture(scope="module")
def kat(golden_dir):
    return np.load(os.path.join(golden_dir, "kat_frame.npz"))


@pytest.fixture(scope="module")
def utts(golden_dir):
    return np.load(os.path.join(golden_dir, "utterances.npz"))


CASES = ["synth_1p5s", "synth_ragged", "exact_fit", "too_short", "silence_dc", "tone_noise"]


def test_filterbank_matches_reference(kat):
    fb = rm.get_mel_filterbanks()
    assert fb.shape == (26, 256)
    assert np.array_equal(fb, kat["filterbank"])          # bit-exact, same float64 formula
    assert int((fb != 0).sum()) == 444
    assert np.array_equal(np.array(rm.mel_bin_edges()), kat["bins"].astype(int))
    assert rm.mel_bin_edges() == [9, 12, 15, 18, 21, 25, 29, 33, 38, 43, 49, 54, 61, 68, 75, 84, 93,
                                  102, 113, 124, 136, 150, 164, 180, 196, 215, 235, 256]


def test_kat_frame(kat):
    fb = rm.get_mel_filterbanks()
    spec = rm.get_spec_mag(kat["frame"])
    # reference FFT is float32 under numpy>=2; float64 oracle agrees to ~1e-6 relative
    np.testing.assert_allclose(spec, kat["spec"], rtol=2e-5, atol=1e-3)
    np.testing.assert_allclose(rm.get_mfcc(kat["frame"], fb), kat["mfcc"], rtol=0, atol=5e-6)
    np.testing.assert_allclose(rm.get_mfcc_from_spec(kat["spec"], fb), kat["mfcc_from_spec"], atol=1e-12)
    np.testing.assert_allclose(rm.lifter_coefs(13), kat["lifter13"], atol=1e-15)
    # survey appendix B.2 literal
    np.testing.assert_allclose(kat["mfcc"][:3], [25.5060315931, -3.3371197123, 0.4348178577], atol=1e-9)


def test_zero_frame_eps_branch(kat):
    fb = rm.get_mel_filterbanks()
    z = rm.get_mfcc(np.zeros(400, np.int16), fb)
    np.testing.assert_allclose(z, kat["mfcc_zero"], atol=1e-12)
    assert abs(z[0] - (-79.8178067)) < 1e-6


def test_dct_matrix_matches_scipy():
    from scipy.fftpack import dct
    x = np.random.default_rng(1).standard_normal((7, 26))
    np.testing.assert_allclose(x @ rm.dct2_ortho_matrix(13, 26).T,
                               dct(x, type=2, norm="ortho", axis=1)[:, :13], atol=1e-13)


@pytest.mark.parametrize("name", CASES)
def test_frame_counts(utts, name):
    pcm = utts[name + "/pcm"]
    assert rm.n_frames(len(pcm)) == int(utts[name + "/n_frames"])
    assert rm.n_outputs(len(pcm)) == utts[name + "/dataset_rows"].shape[0]
    assert rm.split_into_frames(pcm).shape[0] == int(utts[name + "/n_frames"])


def test_frame_count_rule():
    assert rm.n_frames(960000) == 5998 and rm.n_outputs(960000) == 5993
    assert rm.n_frames(160000) == 998 and rm.n_outputs(160000) == 993
    assert rm.n_frames(400) == 0 and rm.n_frames(401) == 1 and rm.n_frames(560) == 1 and rm.n_frames(561) == 2


@pytest.mark.parametrize("name", CASES)
def test_mfcc_and_rows_vs_reference_golden(utts, name):
    pcm = utts[name + "/pcm"]
    fb = rm.get_mel_filterbanks()
    c = rm.mfcc_utterance(pcm, fb)
    ref_c = utts[name + "/mfcc"]
    assert c.shape == ref_c.shape
    if c.shape[0] == 0:
        return
    # float32-FFT reference vs float64 oracle; frames with exact zeros are bit-stable
    np.testing.assert_allclose(c, ref_c, rtol=0, atol=2e-5)
    ds = rm.dataset_features(c)
    np.testing.assert_allclose(ds, utts[name + "/dataset_rows"], rtol=0, atol=5e-5)
    an = rm.analyser_features(c)
    ref_an = utts[name + "/analyser_rows"]
    assert an.shape == ref_an.shape
    finite = np.isfinite(ref_an)
    assert np.array_equal(np.isfinite(an), finite)         # sigma5 == 0 -> nan on both sides
    # z = (c-mu)/sigma5 amplifies the f32-vs-f64 FFT difference when sigma5 is tiny
    win = np.lib.stride_tricks.sliding_window_view(ref_c, 5, axis=0)[: ref_c.shape[0] - 5].std(axis=2)
    tol = 1e-4 + 1e-4 / np.maximum(np.tile(win, 3), 1e-12)
    assert np.all(np.abs(an - ref_an)[finite] <= tol[finite])


def test_loop_port_equals_vectorised(utts):
    fb = rm.get_mel_filterbanks()
    pcm = utts["synth_ragged/pcm"]
    feats = ref_loop.process_pcm(pcm, fb)
    rows = np.array([np.concatenate(f) for f in feats])
    np.testing.assert_allclose(rows, utts["synth_ragged/dataset_rows"], atol=1e-9)
    rec = []

    class Stub(object):
        def predict(self, x):
            rec.append(np.array(x[0]))
            return np.array([0])

    an = ref_loop.LoopAnalyser(Stub(), fb)
    for fr in rm.split_into_frames(pcm):
        an.feed_frame(fr.astype(np.float32))
    np.testing.assert_allclose(np.array(rec), utts["synth_ragged/analyser_rows"], atol=1e-9)


def test_ffn_oracle_frozen(golden_dir, utts):
    g = np.load(os.path.join(golden_dir, "ffn_oracle.npz"))
    w = rm.glorot_ffn(0)
    for k in w:
        assert np.array_equal(w[k], g[k])
    logits, probs = rm.ffn_forward(utts["synth_1p5s/analyser_rows"], w)
    np.testing.assert_allclose(logits, g["logits"], atol=1e-12)
    np.testing.assert_allclose(probs.sum(axis=1), 1.0, atol=1e-12)
    assert np.array_equal(rm.decide(logits), g["labels"])
    assert g["labels"].dtype == np.uint8 and set(np.unique(g["labels"])) <= {0, 1}


def test_ffn_nan_rows_are_nonspeech():
    w = rm.glorot_ffn(0)
    x = np.full((2, 39), np.nan)
    logits, _ = rm.ffn_forward(x, w)
    assert np.all(np.isnan(logits)) and np.array_equal(rm.decide(logits), [0, 0])


@pytest.mark.parametrize("name", CASES)
def test_ref_io_wav_path_matches_reference_process_file(utts, name, tmp_path):
    """oracle/ref_io.py's file path (wav read + dataset rows) against the rows the unmodified reference's
    process_file returned for the same PCM written as a 16 kHz wav (tests/golden/utterances.npz)."""
    from scipy.io import wavfile
    from oracle import ref_io
    pcm = utts[name + "/pcm"]
    path = str(tmp_path / "u.wav")
    wavfile.write(path, 16000, pcm)
    got = rm.dataset_features(rm.mfcc_utterance(ref_io.file_samples(path)))
    want = utts[name + "/dataset_rows"]
    assert got.shape == want.shape
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-5)


def test_ffn_oracle_cross_checked_against_torch_linear():
    """The FFN restatement has no reference execution to pin to (Keras 1 is absent), so a second, independent
    implementation checks it: torch.nn.functional.linear / relu / softmax in float64."""
    import torch
    import torch.nn.functional as F
    w = rm.glorot_ffn(7)
    w["b1"] = np.linspace(-0.3, 0.3, 64).astype(np.float32)       # non-zero biases too
    w["b4"] = np.array([0.1, -0.2, 0.05], dtype=np.float32)
    x = np.random.default_rng(0).standard_normal((257, 39)) * np.array([1.0] * 13 + [3.0] * 13 + [20.0] * 13)
    h = torch.from_numpy(x)
    for i in (1, 2, 3):
        h = F.relu(F.linear(h, torch.from_numpy(w["W%d" % i].astype(np.float64)).T,
                            torch.from_numpy(w["b%d" % i].astype(np.float64))))
    logits_t = F.linear(h, torch.from_numpy(w["W4"].astype(np.float64)).T, torch.from_numpy(w["b4"].astype(np.float64)))
    logits, probs = rm.ffn_forward(x, w)
    np.testing.assert_allclose(logits, logits_t.numpy(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(probs, F.softmax(logits_t, dim=1).numpy(), rtol=1e-12, atol=1e-14)
    assert np.array_equal(rm.decide(logits), (logits_t.argmax(dim=1) == 1).numpy().astype(np.uint8))
