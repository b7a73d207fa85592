"""GPU: ffn_predict on the features the fused VAD kernel returns reproduces that kernel's labels and logits bit for bit,
for every classifier implementation, with the argmax rule and with a decision threshold.

The fused block phase and ffn_tc_rows_kernel run the same tile routine on the same float32 features (fused features
always lie within the kFeatBound* limits, so ffn_predict takes the fp16 tiles on them under impl 2), and rows whose
features are not finite come out NaN with label 0 on both sides."""
import numpy as np
import pytest

import _ffn_bound as fb
import _signals

pytestmark = pytest.mark.gpu

WEIGHTS = ("glorot0", "glorot_x3_bias", "trained")
IMPLS = ("fp32", "tc", "tc16")


@pytest.fixture(scope="module")
def handles():
    import torch
    from vad_b200 import runtime
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    sets = fb.weight_sets()
    hs = {name: runtime.Handle(0, ffn_weights=sets[name]) for name in WEIGHTS}
    yield hs
    for h in hs.values():
        h.close()


@pytest.mark.parametrize("theta", [None, 0.5], ids=["argmax", "threshold"])
@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("name", WEIGHTS)
def test_ffn_predict_on_fused_features_matches_fused(handles, name, impl, theta):
    import torch
    from vad_b200 import batch, runtime
    h = handles[name]
    flat, off, ln = batch.pack_utterances(list(_signals.catalogue().values()))
    pcm = flat.to(h.device)
    plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
    try:
        h.set_ffn_impl(impl)
        h.set_decision_threshold(theta)
        for fm in (runtime.FEAT_ANALYSER, runtime.FEAT_DATASET):
            labels, logits, feats = plan.vad(pcm, want_logits=True, want_feats=True, feat_mode=fm)
            p_labels, p_logits = h.ffn_predict(feats)
            torch.cuda.synchronize()
            labels, logits = labels.cpu().numpy(), logits.cpu().numpy()
            p_labels, p_logits = p_labels.cpu().numpy(), p_logits.cpu().numpy()
            if fm == runtime.FEAT_ANALYSER:
                assert np.isnan(logits).any(), "the catalogue's constant signals give non-finite rows"
            assert np.array_equal(p_labels, labels), (fm, np.nonzero(p_labels != labels)[0][:20].tolist())
            assert np.array_equal(np.isnan(p_logits), np.isnan(logits)), fm
            fin = ~np.isnan(logits)
            differ = np.nonzero((p_logits.view(np.uint32) != logits.view(np.uint32)) & fin)[0]
            assert differ.size == 0, (fm, "rows %s" % np.unique(differ)[:20].tolist())
    finally:
        plan.close()
        h.set_ffn_impl("tc16")
        h.set_decision_threshold(None)
