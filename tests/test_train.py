"""FFN training (SURVEY.md 8f, f4): the device trainer against the float64 restatement of Keras-1 train_on_batch
(oracle/ref_train.py).  CPU part: the oracle's gradients against finite differences, the class-mixing generator.
GPU part: 100 steps at batch 4096 track the oracle's loss within 1e-3 relative; weights round-trip through .npz into
the inference path; the fused feature kernel feeds the trainer end to end."""
import os

import numpy as np
import pytest

from oracle import ref_math as rm, ref_train as rt


def _batch_with_clipped_rows(w, n=23, seed=0):
    """Rows of N(0, 4) and, among them, rows scaled by 60: two labelled with their least likely class (p_true far
    below 1e-7: clipped at the low end) and two with their most likely class (p_true far above 1 - 1e-7: clipped at
    the high end).  Returns x, y and the indices of the clipped rows."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, 39)) * 2
    y = rng.integers(0, 3, n)
    low, high = [3, 11], [7, 17]
    x[low + high] *= 60
    logits, _ = rm.ffn_forward(x, w)
    y[low] = logits[low].argmin(axis=1)
    y[high] = logits[high].argmax(axis=1)
    prob = np.exp(logits - logits.max(axis=1, keepdims=True))
    py = (prob / prob.sum(axis=1, keepdims=True))[np.arange(n), y]
    clipped = np.array(low + high)
    assert np.all(py[low] < 1e-9) and np.all(1.0 - py[high] < 1e-9)
    assert np.all((py > 1e-6) & (py < 1.0 - 1e-6) | np.isin(np.arange(n), clipped))   # the rest far from both ends
    return x, y, clipped


def test_oracle_gradients_match_finite_differences():
    """Every entry of every parameter tensor against central differences of the loss, on a batch whose clipped rows
    (both ends) sit among ordinary rows: the clip passes no gradient, so those rows contribute nothing."""
    w = rm.glorot_ffn(3)
    st = rt.init_state(w)
    x, y, _ = _batch_with_clipped_rows(w)
    loss, g = rt.loss_and_grads(st["p"], x, y)
    h = 1e-6
    p2 = {k: v.copy() for k, v in st["p"].items()}
    for k in rt.KEYS:
        fd = np.empty_like(g[k])
        for idx in np.ndindex(*g[k].shape):
            v = p2[k][idx]
            p2[k][idx] = v + h
            lp, _ = rt.loss_and_grads(p2, x, y)
            p2[k][idx] = v - h
            lm, _ = rt.loss_and_grads(p2, x, y)
            p2[k][idx] = v
            fd[idx] = (lp - lm) / (2 * h)
        err = np.abs(fd - g[k])
        assert np.all(err <= 1e-7 + 1e-5 * np.abs(g[k])), (k, np.unravel_index(err.argmax(), err.shape), err.max())
    # Adadelta's first step: a = (1-rho) g^2, u = g sqrt(eps) / sqrt(a + eps)
    before = {k: v.copy() for k, v in st["p"].items()}
    rt.train_on_batch(st, x, y)
    u = g["W4"] * np.sqrt(1e-8) / np.sqrt(0.05 * g["W4"] ** 2 + 1e-8)
    np.testing.assert_allclose(st["p"]["W4"], before["W4"] - u, atol=1e-15)


def test_oracle_clipped_rows_only_rescale_the_gradient():
    """k clipped rows in a batch of n: the gradient is (n - k) / n times the gradient of the batch without them."""
    w = rm.glorot_ffn(3)
    p = rt.init_state(w)["p"]
    x, y, clipped = _batch_with_clipped_rows(w)
    keep = np.setdiff1d(np.arange(len(y)), clipped)
    _, g = rt.loss_and_grads(p, x, y)
    _, g_kept = rt.loss_and_grads(p, x[keep], y[keep])
    for k in rt.KEYS:
        np.testing.assert_allclose(g[k], g_kept[k] * (len(keep) / len(y)), rtol=1e-12, atol=1e-15, err_msg=k)


def test_mixing_generator_restatements_agree():
    from vad_b200.trainer import mixing_batches
    for sizes in ([50, 30, 20], [500, 300, 200], [7, 7, 7], [1000, 10, 1]):
        o = rt.mixing_order(sizes, np.random.RandomState(1))
        b = list(mixing_batches(sizes, 10, np.random.RandomState(1)))
        b = np.concatenate(b) if b else np.zeros(0, dtype=np.int64)
        assert np.array_equal(b, o[: len(b)]) and len(o) - len(b) < 10
        assert np.all(np.bincount(o, minlength=3) <= np.array(sizes))
        assert len(o) >= sum(sizes) - 3 * len(sizes)          # the reference stops at most a few samples early


def _toy_problem(n, seed):
    """Three separable-ish classes in the 39-dim feature space, scaled like dataset rows after scale_features."""
    rng = np.random.default_rng(seed)
    y = rng.integers(0, 3, n)
    centers = rng.standard_normal((3, 39)) * 0.8
    x = centers[y] + rng.standard_normal((n, 39))
    return x.astype(np.float32), y.astype(np.uint8)


@pytest.mark.gpu
def test_100_steps_track_the_oracle_loss():
    import torch
    from vad_b200 import runtime
    from vad_b200.trainer import FFNTrainer
    h = runtime.Handle()
    w0 = rm.glorot_ffn(11)
    tr = FFNTrainer(h, weights=w0, max_batch=4096)
    st = rt.init_state(w0)
    x, y = _toy_problem(4096 * 4, 5)
    dx, dy = torch.from_numpy(x).to(h.device), torch.from_numpy(y).to(h.device)
    losses, ref_losses = [], []
    for step in range(100):
        lo = (step % 4) * 4096
        n = 4096 if step % 7 else 4001                        # a ragged last tile as well
        losses.append(tr.train_on_batch(dx[lo:lo + n].contiguous(), dy[lo:lo + n].contiguous()))
        ref_losses.append(rt.train_on_batch(st, x[lo:lo + n], y[lo:lo + n]))
    losses, ref_losses = np.array(losses), np.array(ref_losses)
    assert ref_losses[-1] < 0.7 * ref_losses[0]               # it learns
    assert np.all(np.abs(losses - ref_losses) <= 1e-3 * ref_losses), np.abs(losses / ref_losses - 1).max()
    got = tr.weights()
    for k in rt.KEYS:
        assert np.all(np.abs(got[k] - st["p"][k]) <= 2e-3 + 2e-3 * np.abs(st["p"][k])), k
    tr.close()


@pytest.mark.gpu
def test_steps_on_batches_larger_than_the_grid_match_the_oracle():
    """More 128-row tiles than persistent CTAs (every CTA accumulates several tiles in registers), a ragged last tile,
    and a batch smaller than one tile: loss and updated weights after each step against the float64 restatement."""
    import torch
    from vad_b200 import runtime
    from vad_b200.trainer import FFNTrainer
    h = runtime.Handle()
    w0 = rm.glorot_ffn(21)
    n_big = 128 * 148 * 2 + 128 * 17 + 37                     # > 2 tiles per CTA on a 148-SM part, ragged tail
    tr = FFNTrainer(h, weights=w0, max_batch=n_big)
    st = rt.init_state(w0)
    x, y = _toy_problem(n_big, 13)
    dx, dy = torch.from_numpy(x).to(h.device), torch.from_numpy(y).to(h.device)
    for n in (n_big, 37, 128 * 149, n_big):
        loss = tr.train_on_batch(dx[:n].contiguous(), dy[:n].contiguous())
        ref = rt.train_on_batch(st, x[:n], y[:n])
        assert abs(loss - ref) <= 1e-4 * ref, (n, loss, ref)
        got = tr.weights()
        for k in rt.KEYS:
            assert np.all(np.abs(got[k] - st["p"][k]) <= 1e-4 + 1e-3 * np.abs(st["p"][k])), (n, k)
    tr.close()


@pytest.mark.gpu
def test_weights_round_trip_into_the_inference_path(tmp_path):
    import torch
    from vad_b200 import runtime
    from vad_b200.trainer import FFNTrainer
    h = runtime.Handle()
    tr = FFNTrainer(h, seed=4, max_batch=2048)
    x, y = _toy_problem(2048, 9)
    dx, dy = torch.from_numpy(x).to(h.device), torch.from_numpy(y).to(h.device)
    l0, a0 = tr.evaluate(dx, dy)
    for _ in range(150):
        tr.train_on_batch(dx, dy, want_loss=False)
    l1, a1 = tr.evaluate(dx, dy)
    assert l1 < l0 and a1 > max(a0, 0.6)
    path = str(tmp_path / "ffn.npz")
    tr.save(path)
    w = runtime.load_ffn_npz(path)
    h2 = runtime.Handle(ffn_weights=w)                         # vadb200_set_ffn_weights
    for impl in ("tc16", "tc", "fp32"):
        h2.set_ffn_impl(impl)
        _, logits = h2.ffn_predict(x[:500])
        ref, _ = rm.ffn_forward(x[:500], w)
        assert np.all(np.abs(logits.cpu().numpy() - ref) <= 1e-3 + 1e-3 * np.abs(ref)), impl
    with pytest.raises(TypeError):
        tr.train_on_batch(dx.cpu(), dy)
    tr.close()


@pytest.mark.gpu
def test_feature_kernel_feeds_the_trainer(tmp_path):
    """End to end: synthetic 'speech-like' and 'noise-like' wav files -> process_files (device ingest, MODE_DATASET rows,
    scale_rows) -> FeatureStore -> device batches -> train() epoch loop -> a classifier the analyser can load."""
    import torch
    from scipy.io import wavfile
    from vad_b200 import batch, runtime
    from vad_b200.trainer import FFNTrainer, train
    from vad_b200.synth import synth_utterance
    h = runtime.Handle()
    rng = np.random.default_rng(2)
    for cls, name in ((0, "noise"), (1, "speech")):
        d = tmp_path / name
        d.mkdir()
        for i in range(6):
            pcm = synth_utterance(80 + cls, i, 16000 * 4).astype(np.float64)
            if cls == 1:                                       # harmonic content for the 'speech' class
                t = np.arange(pcm.size) / 16000.0
                pcm = 0.3 * pcm + 4000 * np.sin(2 * np.pi * (150 + 20 * i) * t) * (1 + np.sin(2 * np.pi * 3 * t))
            wavfile.write(str(d / ("u%d.wav" % i)), 16000, np.clip(pcm, -32768, 32767).astype(np.int16))
        with batch.FeatureStore(str(tmp_path / name)) as st:
            batch.process_files([str(d)], cls, 100, st, handle=h, verbose=False)
    sources = []
    for cls, name in ((0, "noise"), (1, "speech")):
        xs, ys = batch.load_feature_store(str(tmp_path / name))
        assert np.all(ys == cls) and xs.shape[0] > 2000
        sources.append((torch.from_numpy(np.ascontiguousarray(xs)).to(h.device), cls))
    tr = FFNTrainer(h, seed=1, max_batch=256)
    hist = train(tr, sources, epochs=40, batch_size=256, seed=3, save_prefix=str(tmp_path / "model"), log=None)
    assert hist[-1][1] > 0.9 and hist[-1][0] < hist[0][0], hist[-1]
    assert os.path.isfile(str(tmp_path / "model_full_training.npz"))
    from vad_b200.analyser import FFNClassifier
    clf = FFNClassifier(weights=str(tmp_path / "model_full_training.npz"))
    xs, _ = batch.load_feature_store(str(tmp_path / "speech"))
    assert clf.predict(np.array(xs[:400])).mean() > 0.85
    tr.close()
