"""Decision-tree fit on the device (vadb200_tree_fit / runtime.TreeFitter / trainer.fit_tree): bit for bit against
tests/_ref_tree_fit.py on every CPU spec, the device's own analyser features and an unbounded tree of >= 10 k nodes;
against sklearn wherever tied_nodes == 0, including 500 k rows at the reference hyperparameters; invariance to row
order and stream; the round trip into every classifying path; every error case of the C ABI."""
import ctypes as C

import numpy as np
import pytest

import _ref_tree_fit as R
import _signals
from test_tree_fit_cpu import REF, TIE_FREE, spec

pytestmark = pytest.mark.gpu
sklearn_tree = pytest.importorskip("sklearn.tree")


@pytest.fixture(scope="module")
def handle():
    from oracle import ref_math as rm
    from vad_b200 import runtime
    return runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))


@pytest.fixture(scope="module")
def fitter(handle):
    from vad_b200 import runtime
    return runtime.TreeFitter(handle, 600_000)


def _dev(X, y):
    import torch
    return (torch.from_numpy(np.ascontiguousarray(X, np.float32)).cuda(),
            torch.from_numpy(np.ascontiguousarray(y, np.uint8)).cuda())


def _fit(fitter, X, y, **kw):
    return fitter.fit(*_dev(X, y), **kw)


def _same(a, b):
    assert R.same_tree(a, b), [k for k in R.ARRAYS if not R.same_tree({**a, **{j: b[j] for j in R.ARRAYS if j != k}},
                                                                        b)]
    assert a.get("tied_nodes", b.get("tied_nodes")) == b.get("tied_nodes", a.get("tied_nodes"))


@pytest.mark.parametrize("name", TIE_FREE)
def test_device_equals_oracle_and_sklearn_on_cpu_specs(fitter, name):
    X, y, kw = spec(name)
    t = _fit(fitter, X, y, **kw)
    _same(t, R.fit(X, y, **kw))
    assert t["tied_nodes"] == 0
    _same(t, R.sklearn_arrays(sklearn_tree.DecisionTreeClassifier(random_state=0, **kw).fit(X, y)))


@pytest.mark.parametrize("seed", [0, 1])
def test_device_equals_oracle_with_ties(fitter, seed):
    rng = np.random.default_rng(seed)
    n = 3000
    X = rng.normal(size=(n, 39)).astype(np.float32)
    y = ((X[:, :3].sum(axis=1) + rng.normal(size=n)) > 0).astype(np.int64)
    y[rng.random(n) < 0.1] = 2
    X[:, 30] = X[:, 11]
    t = _fit(fitter, X, y, min_samples_leaf=3)
    o = R.fit(X, y, min_samples_leaf=3)
    assert o["tied_nodes"] > 0
    _same(t, o)


@pytest.fixture(scope="module")
def device_feats(handle):
    """The device's own analyser features of the signal catalogue (finite rows)."""
    from vad_b200 import batch, runtime
    sig = list(_signals.catalogue().values()) + [_signals.constant(8000, 0), _signals.lsb_noise(16000)]
    pcm, offs, lens = batch._upload_16k(sig, handle, 16000)
    plan = runtime.Plan(handle, offs, lens, runtime.MODE_VAD)
    _, _, ft = plan.vad(pcm, want_feats=True)
    X = ft.cpu().numpy()
    return np.ascontiguousarray(X[np.isfinite(X).all(axis=1)])


@pytest.mark.parametrize("kind", ["ref", "three", "no1"])
def test_device_features(fitter, device_feats, kind):
    X = device_feats
    rng = np.random.default_rng(0)
    loud = (X[:, 13] > np.median(X[:, 13])).astype(np.int64)
    y, kw = {"ref": (np.where(rng.random(len(X)) < 0.1, 1 - loud, loud), REF),
             "three": (np.where(X[:, 0] > 1.0, 2, loud), dict(min_samples_leaf=2)),
             "no1": (np.where(loud == 1, 2, 0), dict(max_depth=6))}[kind]
    t = _fit(fitter, X, y, **kw)
    _same(t, R.fit(X, y, **kw))
    if t["tied_nodes"] == 0:
        _same(t, R.sklearn_arrays(sklearn_tree.DecisionTreeClassifier(random_state=0, **kw).fit(X, y)))


@pytest.fixture(scope="module")
def deep_data():
    rng = np.random.default_rng(7)
    n = 200_000
    X = rng.normal(size=(n, 39)).astype(np.float32)
    y = ((X[:, 0] + 0.5 * X[:, 1] + rng.normal(scale=0.7, size=n)) > 0).astype(np.int64)
    return X, y


def test_unbounded_deep_tree_and_invariance(handle, fitter, deep_data):
    import torch
    X, y = deep_data
    kw = dict(min_samples_leaf=1)
    t = _fit(fitter, X, y, **kw)
    depth = np.zeros(len(t["feature"]), np.int64)
    for k in range(len(depth)):
        if t["children_left"][k] >= 0:
            depth[t["children_left"][k]] = depth[t["children_right"][k]] = depth[k] + 1
    assert len(depth) >= 10_000 and depth.max() >= 40
    _same(t, R.fit(X, y, **kw))
    perm = np.random.default_rng(1).permutation(len(y))
    _same(_fit(fitter, X[perm], y[perm], **kw), t)
    side = torch.cuda.Stream()
    x, yy = _dev(X, y)
    torch.cuda.synchronize()
    _same(fitter.fit(x, yy, stream=side, **kw), t)


@pytest.fixture(scope="module")
def big():
    rng = np.random.default_rng(11)
    n = 500_000
    X = rng.normal(size=(n, 39)).astype(np.float32)
    y = ((X[:, :4] @ np.array([1.0, -0.7, 0.5, 0.3]) + rng.normal(scale=1.0, size=n)) > 0).astype(np.int64)
    y[X[:, 9] > 2.0] = 2
    clf = sklearn_tree.DecisionTreeClassifier(random_state=0, **REF).fit(X, y)   # ~45 s on the host: once
    return X, y, clf


def test_500k_reference_hyperparameters_equal_sklearn(fitter, big):
    X, y, clf = big
    t = _fit(fitter, X, y, **REF)
    if t["tied_nodes"] == 0:
        _same(t, R.sklearn_arrays(clf))
    else:   # sklearn may break those ties otherwise; every node above the first tie still matches
        assert t["children_left"].shape[0] > 1000
        assert t["feature"][0] == clf.tree_.feature[0] and t["threshold"][0] == clf.tree_.threshold[0]


def test_round_trip_into_every_path(handle, fitter, device_feats, tmp_path):
    import torch
    from oracle import ref_tree
    from vad_b200 import runtime
    X = device_feats
    y = (X[:, 13] > np.median(X[:, 13])).astype(np.int64)
    y[np.random.default_rng(3).random(len(y)) < 0.1] ^= 1
    t = _fit(fitter, X, y, **REF)
    h = runtime.Handle(0)
    h.set_tree(t)
    labels, proba = h.tree_predict(torch.from_numpy(X).cuda())
    assert np.array_equal(labels.cpu().numpy(), ref_tree.speech(runtime.tree_arrays(t), X))
    runtime.save_tree_npz(str(tmp_path / "t.npz"), t)
    back = runtime.load_tree_npz(str(tmp_path / "t.npz"))
    for k in runtime.TREE_KEYS:
        assert np.array_equal(back[k], runtime.tree_arrays(t)[k])
    from vad_b200 import batch
    sig = list(_signals.catalogue().values())[:4]
    got = batch.vad_batch(sig, handle=h)
    pcm, offs, lens = batch._upload_16k(sig, h, 16000)
    plan = runtime.Plan(h, offs, lens, runtime.MODE_VAD)
    _, _, ft = plan.vad(pcm, want_feats=True)
    want = ref_tree.speech(runtime.tree_arrays(t), ft.cpu().numpy())
    fin = np.isfinite(ft.cpu().numpy()).all(axis=1)
    assert np.array_equal(torch.cat(got).cpu().numpy()[fin], want[fin])


def test_errors_keep_the_previous_result(handle, fitter):
    import torch
    from vad_b200 import _lib, runtime
    lib = handle.lib
    X, y, kw = spec("depth3")
    t = _fit(fitter, X, y, **kw)
    x, yy = _dev(X, y)
    p = _lib.TreeFitParams()
    lib.vadb200_default_tree_fit_params(C.byref(p))
    assert (p.max_depth, p.min_samples_split, p.min_samples_leaf, p.min_impurity_decrease) == (0, 2, 1, 0.0)
    f, st = fitter._f, handle.stream
    bad_x = x.clone()
    bad_x[17, 5] = float("nan")
    bad_y = yy.clone()
    bad_y[3] = 3
    inf_x = x.clone()
    inf_x[0, 0] = float("inf")
    P = lambda t_: C.c_void_p(t_.data_ptr())  # noqa: E731
    cases = [(bad_x, yy, len(y), p), (inf_x, yy, len(y), p), (x, bad_y, len(y), p), (x, yy, 0, p),
             (x, yy, fitter.max_rows + 1, p)]
    for xx, ty, n, pp in cases:
        assert lib.vadb200_tree_fit(f, P(xx), P(ty), n, C.byref(pp), st) == -1
    for field, v in (("min_samples_split", 1), ("min_samples_leaf", 0), ("min_impurity_decrease", -1.0),
                     ("min_impurity_decrease", float("nan"))):
        q = _lib.TreeFitParams()
        lib.vadb200_default_tree_fit_params(C.byref(q))
        setattr(q, field, v)
        assert lib.vadb200_tree_fit(f, P(x), P(yy), len(y), C.byref(q), st) == -1
    assert lib.vadb200_tree_fit(f, None, P(yy), len(y), C.byref(p), st) == -1
    assert lib.vadb200_tree_fit(f, P(x), P(yy), len(y), None, st) == -1
    assert lib.vadb200_tree_fit(None, P(x), P(yy), len(y), C.byref(p), st) == -1
    _same(fitter.result(), t)
    out = C.c_void_p()
    assert lib.vadb200_tree_fitter_create(None, 10, C.byref(out)) == -1 and not out
    assert lib.vadb200_tree_fitter_create(handle._h, 0, C.byref(out)) == -1 and not out
    # fitting never installs a tree; the fitter outlives its handle
    h2 = runtime.Handle(0)
    f2 = runtime.TreeFitter(h2, 1000)
    assert f2.node_count == 0
    assert lib.vadb200_tree_fit_result(f2._f, *([None] * 10)) == -5
    assert lib.vadb200_get_classifier(h2._h) == 0
    f2.fit(x[:1000].contiguous(), yy[:1000].contiguous(), max_depth=2)
    assert lib.vadb200_get_classifier(h2._h) == 0 and f2.node_count > 1
    h2.close()
    f2.close()
    torch.cuda.synchronize()


def test_fit_tree_flow(handle, device_feats, tmp_path):
    import torch
    from vad_b200 import runtime, trainer
    X = torch.from_numpy(device_feats).cuda()
    loud = X[:, 13] > X[:, 13].median()
    Xn = X.clone()
    Xn[:5, 2] = float("nan")
    logs = []
    tree, acc = trainer.fit_tree([(Xn[~loud].contiguous(), 0), (Xn[loud].contiguous(), 1)], handle=handle,
                                 save_path=str(tmp_path / "tree.npz"), log=logs.append)
    assert any("non-finite" in m for m in logs)
    assert 0.5 < acc <= 1.0
    h = runtime.Handle(0)
    h.set_tree(str(tmp_path / "tree.npz"))
    assert h.tree_node_count == tree["feature"].shape[0]
