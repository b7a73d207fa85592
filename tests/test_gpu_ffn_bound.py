"""GPU: every classifier path's logits, entry by entry, against tests/_ffn_bound.py's rounding bound on the kernel's
own float32 inputs, and every label against the decision rule applied to the device's own logits.

Inputs are the features the fused kernel writes (want_feats), the windows' features vad_windows writes, and the rows
given to ffn_predict, so MFCC and feature error play no part and the bound can be tight.  Kernels reached:

* fused_kernel / fused_fe_kernel <2, 2> (ffn_tc16_tile<2>), <2, 1> (ffn_tc_tile<2>), <2, 0> (classify_row / ffn_forward)
  under FEAT_ANALYSER and FEAT_DATASET, on utterances whose last block phase holds 1 to 256 centres, catalogue
  signals and digital silence, with segment ends mid-phase;
* ffn_tc_rows_kernel<2> (ffn_tc16_tile<1>, and its per-tile fall-back to the tf32 blob), ffn_tc_rows_kernel<1>,
  rows_kernel<FfnParams>;
* windows_kernel<FfnParams> (classify_row);
* stream_feed_kernel's classifier, through its logits equalling the fused fp32 path's bit for bit.

Rows whose features are not finite must come out NaN with label 0."""
import hashlib

import numpy as np
import pytest

from oracle import ref_math as rm
from vad_b200.synth import synth_utterance

import _ffn_bound as fb
import _signals

pytestmark = pytest.mark.gpu

SETS = fb.weight_sets()
IMPLS = ("tc16", "tc", "fp32")
SEGMENT_FRAMES = (64, 128, 160, 2048)
FINAL_PHASE = (1, 127, 128, 129, 255, 256, 257)
THETA = 0.5
WORST = {}                       # (entry point, bound impl) -> worst |d| / bound, reported at the end
_BOUNDS = {}                     # the same features recur across segment lengths and implementations


def samples_for_rows(r):
    """PCM length whose utterance has r output rows (r + 5 frames)."""
    return rm.FRAME_SIZE + (r + 4) * rm.FRAME_STEP + 1


def utterances():
    out = []
    for i, c in enumerate(FINAL_PHASE):     # last block phase: c centres, after one phase (252) and a full one (256)
        out.append(synth_utterance(31, i, samples_for_rows(252 + 256 + c)))
    out += [synth_utterance(32, i, samples_for_rows(c)) for i, c in enumerate(FINAL_PHASE)]
    out += list(_signals.catalogue().values())
    mixed = synth_utterance(33, 0, 16000 * 2)
    mixed[6000:9000] = 0                     # digital silence: NaN rows next to valid ones in the same tile
    out += [mixed, np.zeros(8000, np.int16)]
    for u in out:
        assert rm.n_frames(len(u)) > 5
    return [np.ascontiguousarray(u, np.int16) for u in out]


UTTS = utterances()


@pytest.fixture(scope="module")
def handles():
    import torch
    from vad_b200 import runtime
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    hs = {name: runtime.Handle(0, ffn_weights=w) for name, w in SETS.items()}
    yield hs
    for h in hs.values():
        h.close()
    if WORST:
        print("\nworst |d| / bound:")
        for k in sorted(WORST):
            print("  %-34s %-11s %.4f" % (k[0], k[1], WORST[k]))


def bound_impl(name, impl):
    if impl == "fp32":
        return "fp32"
    if impl == "tc16" and fb.tc16_scales(SETS[name])[0]:
        return "tc16"
    return "tc"


def check(entry, name, impl_b, x, logits, labels, theta=None):
    """Logits within the bound, invalid rows NaN / 0, labels = the decision rule on the device's logits."""
    w = SETS[name]
    valid = np.isfinite(x).all(axis=1)
    assert np.all(np.isnan(logits[~valid])) and np.all(labels[~valid] == 0), (entry, name)
    x, lg, lab = x[valid], logits[valid], labels[valid]
    if x.shape[0] == 0:
        return
    key = (name, impl_b, hashlib.blake2b(x.tobytes(), digest_size=16).digest())
    if key not in _BOUNDS:
        _BOUNDS[key] = fb.forward64(x, w)[0][3], fb.ffn_bound(x, w, impl_b)
    ref, bound = _BOUNDS[key]
    err = np.abs(lg.astype(np.float64) - ref)
    bad = np.nonzero(~(err <= bound))[0]
    assert bad.size == 0, "%s %s %s: rows %s exceed the bound (worst |d| / bound %.3g)" % (
        entry, name, impl_b, np.nonzero(valid)[0][np.unique(bad)][:20].tolist(), np.max(err / bound))
    with np.errstate(invalid="ignore", divide="ignore"):
        frac = np.where(bound > 0, err / bound, 0.0)
    k = (entry, impl_b)
    WORST[k] = max(WORST.get(k, 0.0), float(frac.max()))
    if name == "w4_zero":
        assert np.array_equal(lg, np.broadcast_to(w["b4"], lg.shape)), (entry, impl_b)
    if theta is None:
        assert np.array_equal(lab, fb.decide_argmax(lg)), (entry, name, impl_b)
    else:
        want, sure = fb.decide_threshold(lg, theta)
        assert np.array_equal(lab[sure], want[sure]), (entry, name, impl_b)


def set_fe(h, fe):
    if fe:
        h.set_frontend(0.97, "hamming")
        h.set_decision_threshold(THETA)
    else:
        h.set_frontend(0.0, None)
        h.set_decision_threshold(None)


@pytest.mark.parametrize("fe", [False, True], ids=["default", "fe"])
@pytest.mark.parametrize("name", list(SETS))
def test_fused_vad_logits_within_bound(handles, name, fe):
    """Fused kernel, every FFN implementation, both feature recipes, automatic and fixed segment lengths."""
    import torch
    from vad_b200 import batch, runtime
    h = handles[name]
    flat, off, ln = batch.pack_utterances(UTTS)
    pcm = flat.to(h.device)
    set_fe(h, fe)
    try:
        for sf in (0,) + SEGMENT_FRAMES:
            h.set_plan_segment_frames(sf)
            plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
            per_impl = {}
            for impl in IMPLS:
                h.set_ffn_impl(impl)
                for fm in (runtime.FEAT_ANALYSER, runtime.FEAT_DATASET):
                    labels, logits, feats = plan.vad(pcm, want_logits=True, want_feats=True, feat_mode=fm)
                    torch.cuda.synchronize()
                    labels, logits, feats = labels.cpu().numpy(), logits.cpu().numpy(), feats.cpu().numpy()
                    check("fused%s sf=%d" % ("_fe" if fe else "", sf) if sf in (0, 2048) else
                          "fused%s mid-phase" % ("_fe" if fe else ""), name, bound_impl(name, impl),
                          feats, logits, labels, THETA if fe else None)
                    per_impl[(impl, fm)] = logits
            if name == "beyond_ea61":          # tc16 keeps the tf32 path
                for fm in (runtime.FEAT_ANALYSER, runtime.FEAT_DATASET):
                    assert np.array_equal(per_impl[("tc16", fm)].view(np.uint32), per_impl[("tc", fm)].view(np.uint32))
            plan.close()
    finally:
        h.set_plan_segment_frames(0)
        h.set_ffn_impl("tc16")
        set_fe(h, False)


def feature_rows():
    x = np.concatenate([rm.vad_utterance(u, SETS["glorot0"])[1] for u in UTTS[:4]])
    return x[np.isfinite(x).all(axis=1)].astype(np.float32)


FEATS = feature_rows()


def predict_rows(n, wide_tiles):
    """n rows: analyser features, with all-zero, -0, exactly-at-bound, tiny and single-NaN rows spread over the
    tiles, and in each tile of ``wide_tiles`` one row just above the feature bounds (the tf32 fall-back)."""
    rng = np.random.default_rng(n)
    x = FEATS[rng.integers(0, FEATS.shape[0], n)].copy()
    bound = fb.FEAT_BOUND.astype(np.float32)
    special = [np.zeros(39, np.float32), -np.zeros(39, np.float32),
               bound * rng.choice([-1, 1], 39).astype(np.float32),
               (rng.standard_normal(39) * 1e-3).astype(np.float32)]
    nan_row = FEATS[0].copy()
    nan_row[17] = np.nan
    special.append(nan_row)
    for j, row in enumerate(special):
        for t in range((n + 127) // 128):
            i = 128 * t + (37 * j + 11 * t) % 128
            if i < n:
                x[i] = row
    for t in wide_tiles:
        i = min(128 * t + 64, n - 1)
        x[i] = np.nextafter(bound, np.float32(np.inf)) * rng.choice([-1, 1], 39).astype(np.float32)
    return x


ROW_CASES = [(n, ()) for n in (1, 127, 128, 129, 255, 256)] + [(257, (0, 2)), (128 * 5 + 37, (0, 2, 5))]


@pytest.mark.parametrize("name", list(SETS))
def test_ffn_predict_logits_within_bound(handles, name):
    from vad_b200 import runtime  # noqa: F401
    h = handles[name]
    try:
        for n, wide in ROW_CASES:
            x = predict_rows(n, wide)
            got = {}
            for impl in IMPLS:
                h.set_ffn_impl(impl)
                labels, logits = h.ffn_predict(x)
                got[impl] = (labels.cpu().numpy(), logits.cpu().numpy())
            tiles = np.zeros(n, bool)
            for t in wide:
                tiles[128 * t:128 * (t + 1)] = True
            for impl in IMPLS:
                labels, logits = got[impl]
                bi = bound_impl(name, impl)
                if bi == "tc16":               # tiles holding a wide row run on the tf32 blob: tc's logits bit for bit
                    assert np.array_equal(logits[tiles].view(np.uint32), got["tc"][1][tiles].view(np.uint32)), n
                    check("ffn_predict", name, "tc", x[tiles], logits[tiles], labels[tiles])
                    check("ffn_predict", name, bi, x[~tiles], logits[~tiles], labels[~tiles])
                else:
                    check("ffn_predict", name, bi, x, logits, labels)
                if name == "beyond_ea61" and impl == "tc16":
                    assert np.array_equal(logits.view(np.uint32), got["tc"][1].view(np.uint32))
    finally:
        h.set_ffn_impl("tc16")


@pytest.mark.parametrize("name", list(SETS))
def test_vad_windows_logits_within_bound(handles, name):
    from vad_b200 import runtime
    h = handles[name]
    c = np.concatenate([np.lib.stride_tricks.sliding_window_view(rm.mfcc_utterance(u), 5, axis=0).transpose(0, 2, 1)
                        for u in UTTS[:10]]).astype(np.float32)
    for fm in (runtime.FEAT_ANALYSER, runtime.FEAT_DATASET):
        labels, logits, feats = h.vad_windows(c, feat_mode=fm, want_feats=True)
        check("vad_windows", name, "fp32", feats.cpu().numpy(), logits.cpu().numpy(), labels.cpu().numpy())


def test_stream_bank_logits_equal_fused_fp32(handles):
    """The stream kernel's classifier runs ffn_forward's FFMA order; fed the same samples its logits equal the fused
    fp32 path's bit for bit, so the fused check above covers it."""
    from vad_b200 import batch
    from vad_b200.analyser import StreamBank
    h = handles["glorot_x3_bias"]
    n_chunks = 100
    utts = [u[:160 * n_chunks] for u in UTTS if len(u) >= 160 * n_chunks][:8]
    h.set_ffn_impl("fp32")
    try:
        flat, off, ln = batch.pack_utterances(utts)
        from vad_b200 import runtime
        plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
        _, logits, _ = plan.vad(flat.to(h.device), want_logits=True)
        logits = logits.cpu().numpy()
        ro = plan.row_offsets
        bank = StreamBank(len(utts), handle=h)
        lg = np.zeros((len(utts), n_chunks, 3), np.float32)
        for j in range(n_chunks):
            _, lg[:, j] = bank.feed(np.stack([u[160 * j:160 * (j + 1)] for u in utts]), want_logits=True)
        k = n_chunks - 7
        for s in range(len(utts)):
            assert np.array_equal(lg[s, 7:7 + k].view(np.uint32), logits[ro[s]:ro[s] + k].view(np.uint32)), s
        plan.close()
    finally:
        h.set_ffn_impl("tc16")
