"""GPU: the decision-tree classifier (vadb200_set_tree) on every VAD path.  Labels equal sklearn's predict (argmax) or
predict_proba[:, 1] >= threshold on the features the same call returns, probabilities equal float32(predict_proba),
rows with a non-finite feature get label 0 and NaN -- every row, no tolerance.  The fused kernel, tree_predict,
vad_windows, vad_host, FusedAnalyser(TreeClassifier) and the fixed and ragged banks agree bit for bit; switching
classifiers and alternating handles leave the FFN path as it was."""
import numpy as np
import pytest

from oracle import ref_math as rm
from oracle import ref_tree

import _signals
from test_gpu_stream_ragged import catalogue_signals, feed_signals, fixed_labels, offline
from test_gpu_stream_speech import check_utterance

pytestmark = pytest.mark.gpu
sklearn_tree = pytest.importorskip("sklearn.tree")

THETAS = (0.0, 0.3, 0.5, 0.9)
FRONT = {"plain": (0.0, None), "preemph_hamming": (0.97, "hamming")}


@pytest.fixture(scope="module")
def feats():
    """Oracle analyser features of the signal catalogue plus near-silent signals (training rows)."""
    sig = list(_signals.catalogue().values()) + [_signals.constant(8000, 0), _signals.lsb_noise(16000)]
    return np.concatenate([rm.vad_utterance(s, rm.glorot_ffn(0))[1] for s in sig]).astype(np.float32)


def _fit(X, y, seed=0, **kw):
    ok = np.isfinite(X).all(axis=1)
    return sklearn_tree.DecisionTreeClassifier(random_state=seed, **kw).fit(X[ok], y[ok])


@pytest.fixture(scope="module")
def trees(feats):
    X = feats
    rng = np.random.default_rng(0)
    loud = (X[:, 13] > np.nanmedian(X[:, 13])).astype(np.int64)
    noisy = np.where(rng.random(len(X)) < 0.1, 1 - loud, loud)
    Xd = np.concatenate([X * np.float32(1 + 0.2 * k) + rng.normal(size=X.shape).astype(np.float32)
                         for k in range(40)])
    Xd = Xd[np.isfinite(Xd).all(axis=1)]
    music = np.where(X[:, 0] > 1.0, 2, loud)
    t = dict(
        leaf=_fit(X, np.ones(len(X), np.int64)),
        stump=_fit(X, loud, max_depth=1),
        ref=_fit(X, noisy, max_depth=25, min_samples_leaf=20, min_samples_split=22),
        deep=_fit(Xd, rng.integers(0, 2, len(Xd)), seed=1),
        three=_fit(X, music, seed=2, min_samples_leaf=2),
        no1=_fit(X, np.where(loud == 1, 2, 0), seed=3, max_depth=6),
    )
    assert t["deep"].tree_.node_count >= 10000 and t["deep"].tree_.max_depth >= 40
    return t


def _handle(tree=None, fe="plain", th=0.0):
    from vad_b200 import runtime
    h = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    if tree is not None:
        h.set_tree(tree)
    a, w = FRONT[fe]
    h.set_frontend(a, w)
    h.set_decision_threshold(th)
    return h


def _want(clf, X, th):
    """The library's decision, labels and probabilities by class id, for feature rows X (sklearn itself)."""
    fin = np.isfinite(X).all(axis=1)
    Xs = np.where(np.isfinite(X), X, 0).astype(np.float32)
    cls = list(clf.classes_)
    p = clf.predict_proba(Xs)
    if th <= 0:
        lab = clf.predict(Xs) == 1
    else:
        lab = p[:, cls.index(1)] >= np.float64(np.float32(th)) if 1 in cls else np.zeros(len(X), bool)
    pr = np.zeros((len(X), 3), np.float32)
    for k, c in enumerate(cls):
        pr[:, int(c)] = p[:, k].astype(np.float32)
    lab = np.where(fin, lab, False).astype(np.uint8)
    pr[~fin] = np.nan
    return lab, pr


def _check(clf, X, labels, proba, th, rows=slice(None)):
    lab, pr = _want(clf, X, th)
    assert np.array_equal(labels[rows], lab[rows])
    assert np.array_equal(proba[rows], pr[rows], equal_nan=True)


def _batch():
    sig = list(_signals.catalogue().values()) + [_signals.constant(5000, 0), np.zeros(3000, np.int16),
                                                  _signals.lsb_noise(7000)]
    return [s[:len(s) - 37 * i] for i, s in enumerate(sig)]


@pytest.mark.parametrize("fe", sorted(FRONT))
@pytest.mark.parametrize("kind", ["leaf", "stump", "ref", "deep", "three", "no1"])
def test_fused_and_rows_equal_sklearn(trees, kind, fe):
    import torch
    from vad_b200 import batch, runtime
    clf = trees[kind]
    utts = _batch()
    for th in THETAS:
        h = _handle(clf, fe, th)
        assert h.lib.vadb200_get_classifier(h._h) == 2
        assert h.tree_node_count == clf.tree_.node_count and h.tree_depth == clf.tree_.max_depth
        pcm, offs, lens = batch._upload_16k(utts, h, 16000)
        for seg in (0, 64, 160):
            h.set_plan_segment_frames(seg)
            for fm in (runtime.FEAT_ANALYSER, runtime.FEAT_DATASET):
                plan = runtime.Plan(h, offs, lens, runtime.MODE_VAD)
                lab, lg, ft = plan.vad(pcm, want_logits=True, want_feats=True, feat_mode=fm)
                X = ft.cpu().numpy()
                _check(clf, X, lab.cpu().numpy(), lg.cpu().numpy(), th)
                # tree_predict on the fused features: bit for bit
                l2, p2 = h.tree_predict(ft)
                assert torch.equal(l2, lab) and np.array_equal(p2.cpu().numpy(), lg.cpu().numpy(), equal_nan=True)
                if seg == 0:
                    lh = torch.empty_like(lab, device="cpu").pin_memory()
                    gh = torch.empty_like(lg, device="cpu").pin_memory()
                    plan.vad_host(pcm.cpu(), lh, gh, feat_mode=fm)
                    assert torch.equal(lh, lab.cpu())
                    assert np.array_equal(gh.numpy(), lg.cpu().numpy(), equal_nan=True)
        h.close()


@pytest.mark.parametrize("kind", ["ref", "three", "no1"])
def test_windows_and_nonfinite_rows(trees, kind):
    import torch
    from vad_b200 import runtime
    clf = trees[kind]
    h = _handle(clf)
    rng = np.random.default_rng(5)
    win = rng.normal(size=(3000, 5, 13)).astype(np.float32) * 10
    win[::7] = win[::7, :1]                          # a constant window: z-score NaN (feature mode 0)
    win[5, 2, 3] = np.inf
    for th in THETAS:
        h.set_decision_threshold(th)
        for fm in (runtime.FEAT_ANALYSER, runtime.FEAT_DATASET):
            lab, lg, ft = h.vad_windows(win, fm, want_feats=True)
            X = ft.cpu().numpy()
            fin = np.isfinite(X).all(axis=1)
            assert not fin.all()
            # analyser rows with a non-finite z-score are rejected; dataset rows have no such rule (window_features),
            # and sklearn takes no infinite input: those are compared where finite
            _check(clf, X, lab.cpu().numpy(), lg.cpu().numpy(), th, slice(None) if fm == runtime.FEAT_ANALYSER else fin)
        x = rng.normal(size=(5000, 39)).astype(np.float32) * 20
        x[3, 4], x[9, 38] = np.nan, -np.inf
        lab, pr = h.tree_predict(x)
        _check(clf, x, lab.cpu().numpy(), pr.cpu().numpy(), th)
        # against the float64 restatement on the same float32 rows
        xs = np.where(np.isfinite(x), x, 0)
        fin = np.isfinite(x).all(axis=1)
        assert np.array_equal(lab.cpu().numpy()[fin], ref_tree.speech(runtime.tree_arrays(clf), xs, th)[fin])
    h.close()


def test_tree_predict_is_one_launch_in_guard_bands(trees):
    import torch
    h = _handle(trees["deep"])
    n = 1000
    x = torch.randn((n, 39), device="cuda") * 3
    lab = torch.full((n + 64,), 77, dtype=torch.uint8, device="cuda")
    pr = torch.full((n + 64, 3), 77.0, device="cuda")
    c0 = h.lib.vadb200_launch_count()
    from vad_b200._lib import check
    import ctypes as C
    check(h.lib.vadb200_tree_predict(h._h, C.c_void_p(x.data_ptr()), n, C.c_void_p(lab[32:].data_ptr()),
                                     C.c_void_p(pr[32:].data_ptr()), h.stream))
    assert h.lib.vadb200_launch_count() - c0 == 1
    torch.cuda.synchronize()
    assert (lab[:32] == 77).all() and (lab[32 + n:] == 77).all()
    assert (pr[:32] == 77).all() and (pr[32 + n:] == 77).all()
    _check(trees["deep"], x.cpu().numpy(), lab[32:32 + n].cpu().numpy(), pr[32:32 + n].cpu().numpy(), 0.0)
    # graph capture
    g = torch.cuda.CUDAGraph()
    out = torch.empty((n,), dtype=torch.uint8, device="cuda")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            check(h.lib.vadb200_tree_predict(h._h, C.c_void_p(x.data_ptr()), n, C.c_void_p(out.data_ptr()),
                                             C.c_void_p(0), C.c_void_p(s.cuda_stream)))
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, lab[32:32 + n])
    h.close()


def test_switching_and_isolation(trees):
    import torch
    from vad_b200 import batch
    utts = _batch()
    plain = _handle()
    ref_lab, ref_lg = batch.vad_batch(utts, handle=plain, want_logits=True)
    h = _handle(trees["ref"])
    assert h.has_tree and h.has_classifier
    t_lab, t_lg = batch.vad_batch(utts, handle=h, want_logits=True)
    h.clear_tree()
    assert h.lib.vadb200_get_classifier(h._h) == 1 and h.tree_node_count == 0
    lab, lg = batch.vad_batch(utts, handle=h, want_logits=True)
    for a, b in zip(lab + lg, ref_lab + ref_lg):
        assert torch.equal(a, b) if a.dtype == torch.uint8 else np.array_equal(a.cpu().numpy(), b.cpu().numpy(),
                                                                               equal_nan=True)
    h.set_tree(trees["ref"])
    for _ in range(2):                                   # alternate a tree handle and an FFN handle
        a = batch.vad_batch(utts, handle=h, want_logits=True)
        b = batch.vad_batch(utts, handle=plain, want_logits=True)
        for x, y in zip(a[0] + a[1], t_lab + t_lg):
            assert np.array_equal(x.cpu().numpy(), y.cpu().numpy(), equal_nan=True)
        for x, y in zip(b[0] + b[1], ref_lab + ref_lg):
            assert np.array_equal(x.cpu().numpy(), y.cpu().numpy(), equal_nan=True)
    # a malformed tree leaves the handle as it was
    from vad_b200 import _lib
    bad = dict(**{k: v for k, v in __import__("vad_b200.runtime", fromlist=["x"]).tree_arrays(trees["ref"]).items()})
    bad["feature"] = bad["feature"].copy()
    bad["feature"][0] = 40
    with pytest.raises(_lib.VadB200Error):
        h.set_tree(bad)
    assert h.tree_node_count == trees["ref"].tree_.node_count
    a = batch.vad_batch(utts, handle=h)
    assert all(torch.equal(x, y) for x, y in zip(a, t_lab))
    # no classifier: the error stays
    from vad_b200 import runtime
    bare = runtime.Handle(0)
    with pytest.raises(RuntimeError):
        batch.vad_batch(utts, handle=bare)
    bare.set_tree(trees["stump"])
    assert len(batch.speech_segments(utts, handle=bare)) == len(utts)
    assert len(batch.extract_speech(utts, handle=bare)) == len(utts)
    for x in (h, plain, bare):
        x.close()


@pytest.mark.parametrize("fe", sorted(FRONT))
@pytest.mark.parametrize("th", [0.0, 0.5])
def test_banks_emit_vad_batch_rows(trees, fe, th):
    from vad_b200.analyser import StreamBank, TreeClassifier
    h = _handle(trees["ref"], fe, th)
    n = 40
    sig = catalogue_signals(n, 3)
    want_lab, want_lg = offline(h, sig)
    fl, fg = fixed_labels(h, sig)
    for i, s in enumerate(sig):
        k = len(fl[i])
        assert np.array_equal(fl[i], want_lab[i][:k])
        assert np.array_equal(fg[i], want_lg[i][:k], equal_nan=True)
    rng = np.random.default_rng(1)
    for cap, draw in ((160, lambda i: 160), (700, lambda i: int(rng.integers(0, 701))),
                      (2000, lambda i: 2000 if i % 3 == 0 else int(rng.integers(1, 50)))):
        bank = StreamBank(n, handle=h, max_feed_samples=cap)
        labs, lgs = feed_signals(bank, sig, draw, idle=0.2, rng=rng)
        for i in range(n):
            assert np.array_equal(labs[i], want_lab[i])
            assert np.array_equal(lgs[i], want_lg[i], equal_nan=True)
    # classifier= builds the tree handle itself
    tc = TreeClassifier(trees["ref"])
    tc.handle.set_frontend(*FRONT[fe])
    tc.handle.set_decision_threshold(th)
    bank = StreamBank(n, classifier=tc, max_feed_samples=480)
    labs, _ = feed_signals(bank, sig, lambda i: 480)
    assert all(np.array_equal(labs[i], want_lab[i]) for i in range(n))
    h.close()


def test_bank_speech_segments_and_ends(trees):
    from vad_b200.analyser import StreamBank
    S, G, P = 3, 5, 2
    h = _handle(trees["ref"])
    n = 24
    sig = catalogue_signals(n, 4)
    want_lab, _ = offline(h, sig)
    bank = StreamBank(n, handle=h, max_feed_samples=480)
    bank.set_speech(10 * S, 10 * G, 10 * P)
    per = [[[], [], []] for _ in range(n)]
    pos = [0] * n
    while any(p < len(s) for p, s in zip(pos, sig)):
        chunks = [s[p:p + 480] for p, s in zip(pos, sig)]
        pos = [p + len(c) for p, c in zip(pos, chunks)]
        for i, o in enumerate(bank.feed_samples_speech(chunks)):
            for k in range(3):
                per[i][k].append(o[k])
    tails = bank.end_streams(range(n))
    for i in range(n):
        labs, rows, bounds = (np.concatenate(x) for x in per[i])
        lab, _ = check_utterance(S, G, P, labs, rows, bounds, tails[i])   # Plan.speech_segments' smoothing
        assert np.array_equal(lab, want_lab[i])
    h.close()


def test_fused_analyser_tree_classifier(trees):
    from vad_b200.analyser import FusedAnalyser, TreeClassifier
    s = _signals.mixed(16000)
    frames = [s[160 * i:160 * i + 400].astype(np.float32) for i in range((len(s) - 400) // 160)]
    plain = _handle()   # the host path's features come from vad_windows, which needs a classifier on its handle
    for kind in ("ref", "no1", "three"):        # no1 and three hold class 2 (music): both paths raise on it
        dev = FusedAnalyser(classifier=TreeClassifier(trees[kind]))
        host = FusedAnalyser(classifier=trees[kind], handle=plain)
        for f in frames:
            try:
                a = dev.feed_frame(f)
            except AssertionError:
                with pytest.raises(AssertionError):
                    host.feed_frame(f)
                continue
            assert (a is None) == (host.feed_frame(f) is None)
    tc = TreeClassifier(trees["three"])
    x = np.random.default_rng(2).normal(size=(4000, 39)).astype(np.float32) * 5
    assert np.array_equal(tc.predict(x), trees["three"].predict(x))
    assert np.array_equal(tc.predict_proba(x)[:, trees["three"].classes_],
                          trees["three"].predict_proba(x).astype(np.float32))
