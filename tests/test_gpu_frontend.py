"""GPU: the opt-in front end (pre-emphasis, analysis window) and decision threshold through every path that touches
samples or makes a decision, against the float64 oracle at the tolerances of tests/_parity.py."""
import os

import numpy as np
import pytest

from oracle import ref_frontend as rf, ref_math as rm
from vad_b200.synth import synth_utterance

from _parity import LOGIT_ATOL, LOGIT_RTOL, mfcc_close, rows_close
from test_frontend_cpu import threshold_decisive

pytestmark = pytest.mark.gpu

HAMMING = np.hamming(400)
STAGES = [(0.97, None), (0.0, HAMMING), (0.97, HAMMING)]   # each stage alone, then both (catches a wrong order)


@pytest.fixture(scope="module", params=["tc16", "tc", "fp32"])
def fh(request):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vad_b200 import runtime
    w = rm.glorot_ffn(0)
    h = runtime.Handle(0, ffn_weights=w)
    h.set_ffn_impl(request.param)
    yield h, w
    h.close()


@pytest.fixture(scope="module")
def utts(golden_dir):
    return np.load(os.path.join(golden_dir, "utterances.npz"))


def ragged_utts():
    lens = [401, 5, 1041, 16000 + 37, 32003, 561, 25000, 48017]
    return [synth_utterance(17, i, n) for i, n in enumerate(lens)]


def packed_with_garbage(utts):
    """Packed batch whose bytes between utterances are non-zero (the sample before an utterance is never read)."""
    import torch
    from vad_b200 import batch
    flat, off, ln = batch.pack_utterances(utts)
    buf = torch.full((flat.numel() + 16,), -12345, dtype=torch.int16)
    for o, n, u in zip(off, ln, utts):
        buf[o:o + n] = torch.from_numpy(np.asarray(u, dtype=np.int16))
    return buf, off, ln


def check_vad_fe(labels, logits, pcm, w, preemph, window, theta=None, mode="analyser"):
    c, feats, ref_logits, ref_labels = rf.vad_utterance(pcm, w, mode=mode, preemph=preemph, window=window,
                                                        threshold=theta)
    assert labels.shape == ref_labels.shape
    if ref_labels.shape[0] == 0:
        return
    fin = np.isfinite(feats).all(axis=1)
    assert np.all(labels[~fin] == 0)
    assert np.array_equal(np.isfinite(logits).all(axis=1), fin)
    err = np.abs(logits[fin] - ref_logits[fin])
    assert np.all(err <= LOGIT_ATOL + LOGIT_RTOL * np.abs(ref_logits[fin])), err.max()
    if theta is None:
        srt = np.sort(ref_logits[fin], axis=1)
        dec = (srt[:, -1] - srt[:, -2]) > 2 * (LOGIT_ATOL + LOGIT_RTOL * np.abs(srt[:, -1]))
    else:
        dec = threshold_decisive(ref_logits[fin], theta)
    assert np.array_equal(labels[fin][dec], ref_labels[fin][dec])


def frontend(h, preemph, window, theta=None):
    h.set_frontend(preemph, window)
    h.set_decision_threshold(theta)


@pytest.mark.parametrize("preemph,window", STAGES)
def test_golden_utterances_all_modes(fh, utts, preemph, window):
    from vad_b200 import batch
    h, w = fh
    frontend(h, preemph, window)
    try:
        for name in ("synth_1p5s", "synth_ragged", "exact_fit", "too_short", "silence_dc", "tone_noise"):
            pcm = utts[name + "/pcm"]
            c = rf.mfcc_utterance(pcm, preemph=preemph, window=window)
            mf = batch.mfcc_batch([pcm], handle=h)[0].cpu().numpy()
            assert mf.shape == c.shape and (c.shape[0] == 0 or mfcc_close(mf, c))
            ds = batch.mfcc_batch([pcm], deltas=True, handle=h)[0].cpu().numpy()
            assert rows_close(ds, rm.dataset_features(c))
            labels, logits = batch.vad_batch([pcm], handle=h, want_logits=True)
            check_vad_fe(labels[0].cpu().numpy(), logits[0].cpu().numpy(), pcm, w, preemph, window)
    finally:
        frontend(h, 0.0, None)


@pytest.mark.parametrize("preemph,window", STAGES)
def test_ragged_batch_mid_utterance_segments(fh, preemph, window):
    """Segments of 64 frames start mid-utterance (their first frame needs the sample before the segment); the packed
    buffer holds non-zero bytes between utterances (an utterance's first sample has no predecessor)."""
    from vad_b200 import runtime
    h, w = fh
    utts = ragged_utts()
    buf, off, ln = packed_with_garbage(utts)
    frontend(h, preemph, window)
    h.set_plan_segment_frames(64)
    try:
        pcm = buf.to(h.device)
        for mode in (runtime.MODE_MFCC, runtime.MODE_DATASET):
            plan = runtime.Plan(h, off, ln, mode)
            assert plan.segment_count > len(utts)
            out = plan.mfcc(pcm).cpu().numpy()
            for u, r0, r1 in zip(utts, plan.row_offsets[:-1], plan.row_offsets[1:]):
                c = rf.mfcc_utterance(u, preemph=preemph, window=window)
                ref = c if mode == runtime.MODE_MFCC else rm.dataset_features(c)
                assert (mfcc_close if mode == runtime.MODE_MFCC else rows_close)(out[r0:r1], ref)
        plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
        labels, logits, _ = plan.vad(pcm, want_logits=True)
        labels, logits = labels.cpu().numpy(), logits.cpu().numpy()
        for u, r0, r1 in zip(utts, plan.row_offsets[:-1], plan.row_offsets[1:]):
            check_vad_fe(labels[r0:r1], logits[r0:r1], u, w, preemph, window)
    finally:
        h.set_plan_segment_frames(0)
        frontend(h, 0.0, None)


def test_host_pipeline_equals_device_path(fh):
    import torch
    from vad_b200 import batch, runtime
    h, w = fh
    utts = [synth_utterance(11, i, 16000 * (1 + i % 4) + 37 * i) for i in range(24)]
    flat, off, ln = batch.pack_utterances(utts, pin=True)
    frontend(h, 0.97, "hamming", 0.5)
    h.set_plan_segment_frames(64)
    h.set_host_chunk_samples(100000)
    try:
        plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
        dev_labels, dev_logits, _ = plan.vad(flat.to(h.device), want_logits=True)
        logits_host = torch.empty((plan.total_rows, 3), dtype=torch.float32).pin_memory()
        host_labels, _ = plan.vad_host(flat, logits_host=logits_host)
        assert torch.equal(host_labels, dev_labels.cpu())
        assert torch.equal(torch.nan_to_num(logits_host), torch.nan_to_num(dev_logits.cpu()))
        mplan = runtime.Plan(h, off, ln, runtime.MODE_DATASET)
        assert torch.equal(mplan.mfcc_host(flat), mplan.mfcc(flat.to(h.device)).cpu())
    finally:
        h.set_host_chunk_samples(32 << 20)
        h.set_plan_segment_frames(0)
        frontend(h, 0.0, None)


@pytest.mark.parametrize("theta", [0.2, 0.5, 0.8])
def test_thresholds_fused_and_rows(fh, theta):
    import torch
    from vad_b200 import batch
    h, w = fh
    utts = ragged_utts()
    frontend(h, 0.97, "hamming")
    try:
        _, lo0 = batch.vad_batch(utts, handle=h, want_logits=True)
        h.set_decision_threshold(theta)
        assert h.decision_threshold() == pytest.approx(theta)
        labels, logits = batch.vad_batch(utts, handle=h, want_logits=True)
        for u, la, lo, l0 in zip(utts, labels, logits, lo0):
            assert torch.equal(torch.nan_to_num(lo), torch.nan_to_num(l0))      # logits do not depend on theta
            check_vad_fe(la.cpu().numpy(), lo.cpu().numpy(), u, w, 0.97, HAMMING, theta)
        # windows API and classifier.predict duck type
        c = rf.mfcc_utterance(utts[4], preemph=0.97, window=HAMMING)
        win = np.lib.stride_tricks.sliding_window_view(c, 5, axis=0)[: c.shape[0] - 5].transpose(0, 2, 1)
        wl, wlo, wf = h.vad_windows(np.ascontiguousarray(win), want_feats=True)
        ref_lo = rm.ffn_forward(rm.analyser_features(c), w)[0]
        fin = np.isfinite(ref_lo).all(axis=1)
        dec = threshold_decisive(ref_lo[fin], theta)
        assert np.array_equal(wl.cpu().numpy()[fin][dec], rf.decide(ref_lo, theta)[fin][dec])
        x = wf.cpu().numpy()
        pl, plo = h.ffn_predict(x)
        ref_lo = rm.ffn_forward(x, w)[0]
        dec = threshold_decisive(ref_lo, theta)
        assert np.array_equal(pl.cpu().numpy()[dec], rf.decide(ref_lo, theta)[dec])
    finally:
        frontend(h, 0.0, None)


def test_stream_bank_front_end_threshold_and_reset(fh):
    from vad_b200 import batch
    from vad_b200.analyser import StreamBank
    h, w = fh
    n_streams, n_chunks = 40, 50
    L = 160 * n_chunks
    utts = [synth_utterance(41, s, L) for s in range(n_streams)]
    frontend(h, 0.97, "hamming", 0.5)
    try:
        bank = StreamBank(n_streams, handle=h)
        off_labels = batch.vad_batch(utts, handle=h)
        for rnd in range(2):                      # the second round after reset restarts pre-emphasis from 0
            got = np.full((n_streams, n_chunks), 255, np.uint8)
            src = utts if rnd == 0 else [u[::-1].copy() for u in utts]
            for j in range(n_chunks):
                got[:, j] = bank.feed(np.stack([u[160 * j:160 * (j + 1)] for u in src]))
            want = off_labels if rnd == 0 else batch.vad_batch(src, handle=h)
            assert np.all(got[:, :7] == 255)
            for s in range(n_streams):
                k = min(n_chunks - 7, want[s].shape[0])
                assert np.array_equal(got[s, 7:7 + k], want[s].cpu().numpy()[:k])
            bank.reset()
    finally:
        frontend(h, 0.0, None)


def test_per_frame_api_and_analyser(fh):
    from vad_b200._lib import VadB200Error
    from vad_b200.analyser import FusedAnalyser
    h, w = fh
    rng = np.random.default_rng(2)
    fr = (rng.standard_normal((37, 400)) * 1234.5).astype(np.float32)
    try:
        for preemph, window in STAGES:
            frontend(h, preemph, window)
            got = h.spec_frames(fr).cpu().numpy()
            ref = rf.get_spec_mag(rf.preemphasis(fr, preemph), window=window)   # each frame is its own signal
            assert np.max(np.abs(got - ref)) <= 3e-6 * ref.max()
            assert mfcc_close(h.mfcc_frames(fr).cpu().numpy(),
                              rf.get_mfcc(rf.preemphasis(fr, preemph), rm.get_mel_filterbanks(), window=window))
        with pytest.raises(VadB200Error) as e:
            h.spec_frames(fr[:, :320])                       # a window needs 400-sample frames
        assert e.value.code == -1
        frontend(h, 0.97, None)
        short = fr[:, :320].copy()
        ref = rf.get_spec_mag(rf.preemphasis(short, 0.97))
        assert np.max(np.abs(h.spec_frames(short).cpu().numpy() - ref)) <= 3e-6 * ref.max()
        # FusedAnalyser: per-frame MFCC with the front end, external classifier sees the oracle's row
        frontend(h, 0.97, "hamming")
        pcm = synth_utterance(21, 0, 16000)
        frames = rm.split_into_frames(pcm)
        seen = []

        class Stub(object):
            def predict(self, x):
                seen.append(x.copy())
                return np.array([2])

        an = FusedAnalyser(classifier=Stub(), handle=h)
        for f in frames[:5]:
            assert an.feed_frame(f.astype(np.float32)) is None
        with pytest.raises(AssertionError):
            an.feed_frame(frames[5].astype(np.float32))
        c = rf.get_mfcc(rf.preemphasis(frames[:6].astype(np.float32), 0.97), rm.get_mel_filterbanks(), window=HAMMING)
        feats = rm.analyser_features(c)
        assert np.all(np.abs(seen[0][0] - feats[0]) <= 1e-3 + 1e-3 * np.abs(feats[0]))
    finally:
        frontend(h, 0.0, None)


def test_invalid_settings_rejected_and_defaults_restored(fh):
    import torch
    from vad_b200 import batch, runtime
    from vad_b200._lib import VadB200Error
    h, w = fh
    for a in (-0.1, 1.5, float("nan")):
        with pytest.raises(VadB200Error):
            h.set_frontend(a, None)
    bad = np.ones(400)
    bad[7] = np.inf
    with pytest.raises(VadB200Error):
        h.set_frontend(0.5, bad)
    with pytest.raises(ValueError):
        h.set_frontend(0.5, np.ones(399))
    for p in (1.0, 1.5, float("nan")):
        with pytest.raises(VadB200Error):
            h.set_decision_threshold(p)
    assert h.frontend()[0] == 0.0 and h.frontend()[1] is None and h.decision_threshold() is None
    utts = ragged_utts()
    fresh = runtime.Handle(0, ffn_weights=w)
    fresh.set_ffn_impl(h.ffn_impl)
    want = batch.vad_batch(utts, handle=fresh, want_logits=True)
    want_mf = batch.mfcc_batch(utts, deltas=True, handle=fresh)
    h.set_frontend(0.97, "hamming")
    h.set_decision_threshold(0.3)
    a, win = h.frontend()
    assert a == pytest.approx(0.97) and np.array_equal(win, np.hamming(400).astype(np.float32))
    batch.vad_batch(utts, handle=h)
    h.set_frontend(0.0, None)
    h.set_decision_threshold(None)
    got = batch.vad_batch(utts, handle=h, want_logits=True)
    got_mf = batch.mfcc_batch(utts, deltas=True, handle=h)
    for x, y in zip(want[0] + want[1] + want_mf, got[0] + got[1] + got_mf):
        assert torch.equal(torch.nan_to_num(x), torch.nan_to_num(y))
    fresh.close()


def test_process_files_through_a_front_end_handle(fh, tmp_path):
    from scipy.io import wavfile
    from vad_b200 import batch
    h, w = fh
    utts = [synth_utterance(51, i, n) for i, n in enumerate((16000, 24011, 9000))]
    for i, u in enumerate(utts):
        wavfile.write(str(tmp_path / ("f%d.wav" % i)), 16000, u)
    rows = []

    class Sink(object):
        def writerow(self, r):
            rows.append(r)

        def writerows(self, rs):
            rows.extend(rs)

    frontend(h, 0.97, "hamming")
    try:
        n = batch.process_files([str(tmp_path)], 0, 10, Sink(), handle=h, files_per_step=10, verbose=False)
    finally:
        frontend(h, 0.0, None)
    got = np.array([[float(v) for v in r] for r in rows])
    assert n == got.shape[0]
    order = [int(os.path.basename(f)[1:-4]) for f in batch.list_audio_files([str(tmp_path)], 10)]
    groups = [rm.dataset_features(rf.mfcc_utterance(utts[i], preemph=0.97, window=HAMMING)) for i in order]
    want = np.concatenate(rm.scale_features(groups)[0])
    assert got.shape == (want.shape[0], 40)
    assert np.all(np.abs(got[:, :39] - want) <= 1e-3 + 1e-3 * np.abs(want))
