"""GPU: the signal catalogue of tests/_signals.py -- samples on the int16 rails, full-scale tones, a chirp, band-limited
noise, LSB-level audio and a mixed utterance -- through the fused kernel (every mode, default and front-end variants,
every legal segment size), the stream kernel, the per-frame kernel and the host pipeline, plus caller FFN rows far
beyond the MFCC feature range, under all three FFN implementations, against the float64 oracle at the tolerances of
tests/_parity.py."""
import numpy as np
import pytest

from oracle import ref_frontend as rf, ref_math as rm, ref_train as rt

import _signals
from _parity import mfcc_close, rows_close, decisive_rows, LOGIT_ATOL, LOGIT_RTOL
from test_frontend_cpu import threshold_decisive
from test_gpu_frontend import packed_with_garbage

pytestmark = pytest.mark.gpu

CAT = _signals.catalogue()
NAMES = list(CAT)
UTTS = list(CAT.values())
W = rm.glorot_ffn(0)
HAMMING = np.hamming(400)
# name -> (pre-emphasis, window, threshold on p(voiced)); the last window is int16-scaled (a plausible caller
# mistake), which lifts log E about 30 bits past the range the tc16 feature bounds were derived for
FRONT_ENDS = {
    "default": (0.0, None, None),
    "pre_hamming": (0.97, HAMMING, None),
    "pre_hamming_thr": (0.97, HAMMING, 0.5),
    "pre_hamming_int16": (0.97, HAMMING * 32768.0, None),
}
SEGMENT_FRAMES = list(range(64, 2049, 32))          # every legal vadb200_set_plan_segment_frames value


@pytest.fixture(scope="module", params=["tc16", "tc", "fp32"])
def fh(request):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vad_b200 import runtime
    h = runtime.Handle(0, ffn_weights=W)               # private handle: nothing here touches the default one
    h.set_ffn_impl(request.param)
    yield h
    h.close()


def set_fe(h, key):
    preemph, window, theta = FRONT_ENDS[key]
    h.set_frontend(preemph, window)
    h.set_decision_threshold(theta)


def checked(key):
    """Catalogue indices held to the oracle under front end ``key`` (all of them, less the windowed float32 floor)."""
    win = FRONT_ENDS[key][1]
    return [i for i, n in enumerate(NAMES) if win is None or n not in _signals.WINDOWED_FLOAT32_FLOOR]


_ORACLE = {}


def oracle(i, key, mode="analyser", pcm=None):
    """rf.vad_utterance of catalogue entry i (or of ``pcm``) under front end ``key``: (c, feats, logits, labels)."""
    preemph, window, theta = FRONT_ENDS[key]
    if pcm is not None:
        return rf.vad_utterance(pcm, W, mode=mode, preemph=preemph, window=window, threshold=theta)
    k = (i, key, mode)
    if k not in _ORACLE:
        _ORACLE[k] = rf.vad_utterance(UTTS[i], W, mode=mode, preemph=preemph, window=window, threshold=theta)
    return _ORACLE[k]


def check_decisions(labels, logits, ref_feats, ref_logits, ref_labels, theta):
    """NaN rows agree exactly (label 0), finite logits within tolerance, labels equal on decisive rows."""
    assert labels.shape == ref_labels.shape and logits.shape == ref_logits.shape
    fin = np.isfinite(ref_feats).all(axis=1)
    assert np.all(ref_labels[~fin] == 0) and np.all(labels[~fin] == 0)
    assert np.array_equal(np.isfinite(logits).all(axis=1), fin)
    err = np.abs(logits[fin] - ref_logits[fin])
    assert np.all(err <= LOGIT_ATOL + LOGIT_RTOL * np.abs(ref_logits[fin])), err.max()
    dec = decisive_rows(ref_logits[fin]) if theta is None else threshold_decisive(ref_logits[fin], theta)
    assert np.array_equal(labels[fin][dec], ref_labels[fin][dec])


def check_feats(feats, c, ref_feats, mode):
    if mode == "dataset":
        assert rows_close(feats, ref_feats)
        return
    # a row is NaN when any coefficient's sigma5 is 0; which of its entries come out NaN is left to rounding
    fin = np.isfinite(ref_feats).all(axis=1)
    assert np.array_equal(np.isfinite(feats).all(axis=1), fin)
    sig = np.lib.stride_tricks.sliding_window_view(c, 5, axis=0)[: c.shape[0] - 5].std(axis=2)[fin]
    tol = 3e-4 + 2e-4 / np.maximum(np.tile(sig, 3), 1e-12)   # z = (c - mu) / sigma5 amplifies MFCC error
    assert np.all(np.abs(feats[fin] - ref_feats[fin]) <= tol)


def run_all_modes(h, pcm, off, ln):
    """MODE_MFCC, MODE_DATASET and MODE_VAD (both feature recipes, logits and features) of one packed batch."""
    from vad_b200 import runtime
    out = {}
    for mode in (runtime.MODE_MFCC, runtime.MODE_DATASET):
        plan = runtime.Plan(h, off, ln, mode)
        out[mode] = ((plan.mfcc(pcm),), plan.row_offsets)
    plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
    for fm in (runtime.FEAT_ANALYSER, runtime.FEAT_DATASET):
        out[("vad", fm)] = (plan.vad(pcm, want_logits=True, want_feats=True, feat_mode=fm), plan.row_offsets)
    return out


@pytest.mark.parametrize("key", list(FRONT_ENDS))
def test_packed_catalogue_every_mode(fh, key):
    """One ragged batch of the whole catalogue (garbage between utterances).  Front ends run with 64-frame segments,
    so segments continue mid-utterance across full-scale samples."""
    from vad_b200 import runtime
    h = fh
    buf, off, ln = packed_with_garbage(UTTS)
    set_fe(h, key)
    h.set_plan_segment_frames(0 if key == "default" else 64)
    try:
        out = run_all_modes(h, buf.to(h.device), off, ln)
    finally:
        h.set_plan_segment_frames(0)
        set_fe(h, "default")
    theta = FRONT_ENDS[key][2]
    (mf,), ro = out[runtime.MODE_MFCC]
    (ds,), rd = out[runtime.MODE_DATASET]
    mf, ds = mf.cpu().numpy(), ds.cpu().numpy()
    for i in checked(key):
        c = oracle(i, key)[0]
        assert mfcc_close(mf[ro[i]:ro[i + 1]], c), NAMES[i]
        assert rows_close(ds[rd[i]:rd[i + 1]], rm.dataset_features(c)), NAMES[i]
    for fm, mode in ((runtime.FEAT_ANALYSER, "analyser"), (runtime.FEAT_DATASET, "dataset")):
        (labels, logits, feats), rv = out[("vad", fm)]
        labels, logits, feats = labels.cpu().numpy(), logits.cpu().numpy(), feats.cpu().numpy()
        for i in checked(key):
            c, ref_feats, ref_logits, ref_labels = oracle(i, key, mode)
            r0, r1 = rv[i], rv[i + 1]
            try:
                check_decisions(labels[r0:r1], logits[r0:r1], ref_feats, ref_logits, ref_labels, theta)
                check_feats(feats[r0:r1], c, ref_feats, mode)
            except AssertionError as e:
                raise AssertionError("%s (%s): %s" % (NAMES[i], mode, e))


@pytest.mark.parametrize("key", ["default", "pre_hamming"])
def test_every_segment_size_is_byte_identical(fh, key):
    """The segment length changes where segments start (Segment::cont carries the sample before a segment into the
    front end), never a result: every legal length gives the automatic plan's bytes."""
    import torch
    h = fh
    buf, off, ln = packed_with_garbage(UTTS)
    pcm = buf.to(h.device)
    set_fe(h, key)
    try:
        want = run_all_modes(h, pcm, off, ln)
        for sf in SEGMENT_FRAMES:
            h.set_plan_segment_frames(sf)
            got = run_all_modes(h, pcm, off, ln)
            for k, (v, _) in want.items():
                for a, b in zip(v, got[k][0]):
                    assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), (sf, k)
    finally:
        h.set_plan_segment_frames(0)
        set_fe(h, "default")


@pytest.mark.parametrize("key", ["default", "pre_hamming_thr"])
def test_stream_bank_equals_fused_and_oracle(fh, key):
    """StreamBank fed the catalogue (first second of each entry) in 10 ms chunks: labels equal the offline fused
    kernel's, before and after reset(); sampled streams' logits against the oracle."""
    from vad_b200 import batch
    from vad_b200.analyser import StreamBank
    h = fh
    n_chunks = 100
    L = 160 * n_chunks
    utts = [u[:L].copy() for u in UTTS]
    n = len(utts)
    theta = FRONT_ENDS[key][2]
    set_fe(h, key)
    try:
        off_labels = [x.cpu().numpy() for x in batch.vad_batch(utts, handle=h)]
        bank = StreamBank(n, handle=h)
        for rnd in range(2):                       # the second round runs after reset()
            got = np.full((n, n_chunks), 255, np.uint8)
            lg = np.zeros((n, n_chunks, 3), np.float32)
            for j in range(n_chunks):
                got[:, j], lg[:, j] = bank.feed(np.stack([u[160 * j:160 * (j + 1)] for u in utts]), want_logits=True)
            assert np.all(got[:, :7] == 255)
            k = n_chunks - 7
            for s in range(n):
                assert np.array_equal(got[s, 7:7 + k], off_labels[s][:k]), NAMES[s]
            for s in [i for i in checked(key) if NAMES[i] in ("clipped_noise", "square_nyquist", "tone_100_hop_periodic",
                                                               "impulse_train", "lsb_square", "mixed")]:
                _, ref_feats, ref_logits, ref_labels = oracle(None, key, pcm=utts[s])
                check_decisions(got[s, 7:7 + k], lg[s, 7:7 + k], ref_feats[:k], ref_logits[:k], ref_labels[:k], theta)
            bank.reset()
    finally:
        set_fe(h, "default")


def resolvable_in_float32(fr, c):
    """Frames whose MFCCs a float32 FFT (numpy's complex64 path) puts within half the tolerance.  512-sample frames are
    not zero-padded: a constant, the Nyquist square or a bin-centred tone then leaves bins that are 0 in exact
    arithmetic or hold only the int16 rounding noise 120 dB down, and their log energy is float32 rounding alone."""
    import scipy.fft
    X = scipy.fft.fft(fr.astype(np.float32), rm.FFT_N, axis=-1)[:, :rm.FFT_N // 2] / np.float32(rm.FFT_N)
    c32 = rm.get_mfcc_from_spec((X.real ** 2 + X.imag ** 2).astype(np.float64), rm.get_mel_filterbanks())
    return np.all(np.abs(c32 - c) <= 0.5 * (1e-4 + 1e-4 * np.abs(c)), axis=1)


def test_per_frame_api_on_catalogue_frames(fh):
    """spec_frames / mfcc_frames on float frames cut from the catalogue, the same normalised to [-1, 1], and scaled to
    +-1e5 (beyond int16), at frame lengths 400, 399, 320 and 512."""
    h = fh
    fb = rm.get_mel_filterbanks()
    for n in (400, 399, 320, 512):
        base = np.stack([u[s:s + n] for u in UTTS for s in (0, 4321, 9000)]).astype(np.float64)
        for scale in (1.0, 1.0 / 32768.0, 1e5 / 32768.0):
            fr = (base * scale).astype(np.float32)
            spec = h.spec_frames(fr).cpu().numpy()
            ref = rm.get_spec_mag(fr)
            assert np.all(np.abs(spec - ref) <= 3e-6 * ref.max(axis=1, keepdims=True)), (n, scale)
            c = rm.get_mfcc(fr, fb)
            held = resolvable_in_float32(fr, c)
            assert held.mean() > 0.8, (n, scale)
            assert mfcc_close(h.mfcc_frames(fr).cpu().numpy()[held], c[held]), (n, scale)


@pytest.mark.parametrize("key", ["default", "pre_hamming_thr"])
def test_host_pipeline_byte_equal_to_device(fh, key):
    import torch
    from vad_b200 import batch, runtime
    h = fh
    flat, off, ln = batch.pack_utterances(UTTS, pin=True)
    set_fe(h, key)
    h.set_plan_segment_frames(64)
    h.set_host_chunk_samples(100000)               # chunks end inside utterances
    try:
        plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
        for fm in (runtime.FEAT_ANALYSER, runtime.FEAT_DATASET):
            dev_labels, dev_logits, _ = plan.vad(flat.to(h.device), want_logits=True, feat_mode=fm)
            logits_host = torch.empty((plan.total_rows, 3), dtype=torch.float32).pin_memory()
            host_labels, _ = plan.vad_host(flat, logits_host=logits_host, feat_mode=fm)
            assert torch.equal(host_labels, dev_labels.cpu())
            assert torch.equal(logits_host.view(torch.uint8), dev_logits.cpu().view(torch.uint8))
        for mode in (runtime.MODE_MFCC, runtime.MODE_DATASET):
            mplan = runtime.Plan(h, off, ln, mode)
            assert torch.equal(mplan.mfcc_host(flat).view(torch.uint8), mplan.mfcc(flat.to(h.device)).cpu().view(torch.uint8))
    finally:
        h.set_host_chunk_samples(32 << 20)
        h.set_plan_segment_frames(0)
        set_fe(h, "default")


# ---- caller FFN rows beyond the MFCC feature range ------------------------------------------------------
ROW_SCALES = (1e2, 1e3, 1e4, 3e4, 1e5, 1e6)


def wide_rows():
    """(name, rows [n, 39] float32): N(0,1) s, then normal rows with one entry of 7e4 in one feature group."""
    rng = np.random.default_rng(11)
    out = [("N(0,1) x %g" % s, (rng.standard_normal((1000, 39)) * s).astype(np.float32)) for s in ROW_SCALES]
    for g, group in enumerate(("c", "d1", "d2")):
        x = rng.standard_normal((300, 39)).astype(np.float32)
        x[np.arange(300), 13 * g + rng.integers(0, 13, 300)] = 7e4
        out.append(("one %s entry of 7e4" % group, x))
    # in-range rows sharing 128-row tiles with a few wide ones, and tiles with none
    x = rng.standard_normal((1000, 39)).astype(np.float32) * 100
    x[::97, 30] = -7e4
    x[640:] = rng.standard_normal((360, 39)) * 100
    out.append(("mixed tiles", x))
    return out


@pytest.fixture(scope="module")
def trained_weights():
    """A few hundred oracle Adadelta steps from glorot(0) on scaled dataset rows of the catalogue."""
    rows = [rm.dataset_features(rm.mfcc_utterance(u)) for u in UTTS]
    x = np.concatenate(rm.scale_features(rows)[0])
    y = (x[:, 0] > 0).astype(np.int64) + (x[:, 14] > 0.5)
    st = rt.init_state(rm.glorot_ffn(0))
    rng = np.random.default_rng(5)
    for _ in range(300):
        idx = rng.integers(0, x.shape[0], 256)
        rt.train_on_batch(st, x[idx], y[idx])
    return {k: v.astype(np.float32) for k, v in st["p"].items()}


def rounding_reach(x, w):
    """First-order estimate of the logits' rounding error in an evaluation whose products keep about 22 significant
    bits and sum in fp32 (FFMA, and the tf32 and fp16 hi/lo splits): each layer adds 2^-20 (|W| |h| + |b|) on its
    active units and passes the error before it on through |W|.  A logit whose estimate exceeds the tolerance comes
    out of a cancellation no float32 evaluation resolves to it; at every row scale that is roughly half the rows."""
    u = 2.0 ** -20
    h = np.asarray(x, dtype=np.float64)
    e = np.zeros_like(h)
    for i in (1, 2, 3, 4):
        Wi, bi = w["W%d" % i].astype(np.float64), w["b%d" % i].astype(np.float64)
        z = h @ Wi + bi
        e = e @ np.abs(Wi) + u * (np.abs(h) @ np.abs(Wi) + np.abs(bi))
        if i < 4:
            e = np.where(z > 0, e, 0.0)
            h = np.maximum(z, 0.0)
    return e


@pytest.mark.parametrize("weights", ["glorot", "trained"])
def test_ffn_rows_beyond_feature_range(fh, trained_weights, weights):
    """ffn_predict, FFNClassifier.predict and FFNTrainer.evaluate on caller rows far beyond the MFCC feature bounds the
    tc16 scales were chosen for.  Every row gets finite logits.  Rows whose logits float32 can resolve (rounding_reach
    within the tolerance) are held to the logit tolerance and their decisive labels to the oracle's.  Under tc16 a tile holding a wide row runs the tf32 tile: its logits equal the tc path's bit for bit."""
    import torch
    from vad_b200 import runtime
    from vad_b200.analyser import FFNClassifier
    from vad_b200.trainer import FFNTrainer
    w = W if weights == "glorot" else trained_weights
    hh = runtime.Handle(0, ffn_weights=w)
    hh.set_ffn_impl(fh.ffn_impl)
    trainer = FFNTrainer(handle=hh, weights=w)
    try:
        for name, x in wide_rows():
            ref_logits = rm.ffn_forward(x, w)[0]
            labels, logits = hh.ffn_predict(x)
            labels, logits = labels.cpu().numpy(), logits.cpu().numpy()
            bad = ~np.isfinite(logits).all(axis=1)
            assert not bad.any(), "%s: %d rows with non-finite logits" % (name, bad.sum())
            tol = LOGIT_ATOL + LOGIT_RTOL * np.abs(ref_logits)
            held = np.all(rounding_reach(x, w) <= tol, axis=1)
            assert held.mean() > 0.3, name
            err = np.abs(logits - ref_logits)[held]
            assert np.all(err <= tol[held]), "%s: worst err / tol %.3g" % (name, (err / tol[held]).max())
            dec = held & decisive_rows(ref_logits)
            assert np.array_equal(labels[dec], rm.decide(ref_logits)[dec]), name
            assert np.array_equal(FFNClassifier(handle=hh).predict(x)[dec], rm.decide(ref_logits)[dec]), name
            xd = torch.from_numpy(x[dec]).to(hh.device)
            yd = torch.from_numpy(np.argmax(ref_logits[dec], axis=1).astype(np.uint8)).to(hh.device)
            loss, acc = trainer.evaluate(xd, yd)
            assert np.isfinite(loss) and round(acc * dec.sum()) == dec.sum(), (name, loss, acc)
            if fh.ffn_impl == 2:
                hh.set_ffn_impl("tc")
                tc_logits = hh.ffn_predict(x)[1].cpu().numpy()
                hh.set_ffn_impl("tc16")
                wide = np.abs(x) > np.repeat([1353.0, 2706.0, 5416.0], 13)
                tiles = np.repeat(np.add.reduceat(wide.any(axis=1), np.arange(0, x.shape[0], 128)) > 0, 128)[:x.shape[0]]
                assert np.array_equal(logits[tiles], tc_logits[tiles]), name
    finally:
        trainer.close()
        hh.close()
