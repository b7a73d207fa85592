"""Decision-tree classifier without a GPU: oracle/ref_tree.py against sklearn, and the library's own tree conversion
(vad_b200/csrc/vad_tree.h, compiled with g++ by tests/emul/emul_tree.cpp) walked on the CPU against sklearn -- on
random rows, on every threshold's float32 neighbours, on hand-made and infinite thresholds -- plus every malformed
tree it must reject."""
import ctypes as C
import os
import pickle
import subprocess

import numpy as np
import pytest

from oracle import ref_tree
from vad_b200 import _lib, runtime

sklearn_tree = pytest.importorskip("sklearn.tree")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL = os.path.join(ROOT, "tests", "emul")
SO = os.path.join(EMUL, "libvademul_tree.so")
_P = C.c_void_p


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(EMUL, "emul_tree.cpp")
    deps = [src, os.path.join(ROOT, "vad_b200", "csrc", "vad_tree.h")]
    if not os.path.isfile(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO, src])
    lib = C.CDLL(SO)
    lib.emul_tree_convert.argtypes = [C.c_longlong] + [_P] * 6 + [C.c_int] + [_P] * 5 + [C.c_int]
    lib.emul_tree_predict.argtypes = [C.c_longlong] + [_P] * 6 + [C.c_int, _P, C.c_longlong, C.c_float, _P, _P]
    return lib


def _ptrs(a):
    return [a[k].ctypes.data_as(_P) for k in runtime.TREE_KEYS]


def convert(lib, a):
    n = a["children_left"].shape[0]
    t = np.zeros(n, np.float32)
    fl = np.zeros(n, np.uint32)
    leaves = np.zeros((n, 5), np.float64)
    depth = C.c_int()
    err = C.create_string_buffer(256)
    rc = lib.emul_tree_convert(n, *_ptrs(a), int(a["classes"].size), t.ctypes.data_as(_P), fl.ctypes.data_as(_P),
                               leaves.ctypes.data_as(_P), C.byref(depth), err, 256)
    return rc, err.value.decode(), t, fl, leaves, depth.value


def emul_predict(lib, a, X, th=0.0):
    X = np.ascontiguousarray(X, dtype=np.float32)
    m = X.shape[0]
    labels = np.zeros(m, np.uint8)
    proba = np.zeros((m, 3), np.float32)
    rc = lib.emul_tree_predict(a["children_left"].shape[0], *_ptrs(a), int(a["classes"].size), X.ctypes.data_as(_P),
                               m, float(th), labels.ctypes.data_as(_P), proba.ctypes.data_as(_P))
    assert rc == 0
    return labels, proba


def fitted(seed, n=4000, classes=(0, 1), **kw):
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(n, 39)).astype(np.float32) * rng.uniform(0.1, 10, size=39).astype(np.float32)
    y = np.asarray(classes)[rng.integers(0, len(classes), n)]
    y = np.where(X[:, 3] + 0.3 * X[:, 7] > 0, y, np.asarray(classes)[0]) if len(classes) > 1 else y
    clf = sklearn_tree.DecisionTreeClassifier(random_state=seed, **kw).fit(X, y)
    return clf, X


TREES = [
    dict(seed=1, max_depth=1),
    dict(seed=2, max_depth=25, min_samples_leaf=20, min_samples_split=22),
    dict(seed=3),
    dict(seed=4, classes=(0, 1, 2), min_samples_leaf=3),
    dict(seed=5, classes=(0, 2), min_samples_leaf=5),
    dict(seed=6, classes=(1, 2), max_depth=8),
]


def neighbours(clf, X):
    """Rows that put one feature exactly at, one ulp below and one ulp above each threshold's float32 image."""
    t = clf.tree_
    inner = np.flatnonzero(t.children_left != -1)
    rows = []
    for i in inner:
        t32 = np.float32(t.threshold[i])
        for v in (t32, np.nextafter(t32, np.float32(-np.inf)), np.nextafter(t32, np.float32(np.inf))):
            r = X[i % X.shape[0]].copy()
            r[t.feature[i]] = v
            rows.append(r)
    return np.asarray(rows, np.float32)


@pytest.mark.parametrize("spec", TREES, ids=lambda s: "seed%d" % s["seed"])
def test_oracle_equals_sklearn(spec):
    spec = dict(spec)
    clf, X = fitted(spec.pop("seed"), **spec)
    a = runtime.tree_arrays(clf)
    for rows in (X, neighbours(clf, X)):
        assert np.array_equal(ref_tree.apply(a, rows), clf.apply(rows))
        assert np.array_equal(ref_tree.predict(a, rows), clf.predict(rows))
        assert np.array_equal(ref_tree.predict_proba(a, rows), clf.predict_proba(rows))


@pytest.mark.parametrize("spec", TREES, ids=lambda s: "seed%d" % s["seed"])
def test_emulated_layout_equals_sklearn(emul, spec):
    spec = dict(spec)
    clf, X = fitted(spec.pop("seed"), **spec)
    a = runtime.tree_arrays(clf)
    rng = np.random.default_rng(9)
    rows = np.concatenate([X, neighbours(clf, X), rng.normal(size=(2000, 39)).astype(np.float32) * 5])
    cls = list(clf.classes_)
    p64 = clf.predict_proba(rows)
    for th in (0.0, 0.3, 0.5, 0.9):
        labels, proba = emul_predict(emul, a, rows, th)
        if th <= 0:
            want = clf.predict(rows) == 1
        else:
            want = p64[:, cls.index(1)] >= np.float64(np.float32(th)) if 1 in cls else np.zeros(len(rows), bool)
        assert np.array_equal(labels, want.astype(np.uint8))
        for k, c in enumerate(cls):
            assert np.array_equal(proba[:, c], p64[:, k].astype(np.float32))
        for c in set(range(3)) - set(cls):
            assert not proba[:, c].any()


def test_layout_is_breadth_first_with_adjacent_siblings(emul):
    clf, _ = fitted(3)
    a = runtime.tree_arrays(clf)
    rc, err, t, fl, leaves, depth = convert(emul, a)
    assert rc == 0, err
    assert depth == clf.tree_.max_depth
    left, feat = fl >> 6, fl & 63
    idx = np.arange(t.size)
    leaf = left == idx
    assert leaf.sum() == clf.tree_.n_leaves
    assert np.all(np.isinf(t[leaf])) and np.all(feat[leaf] == 0)
    inner = ~leaf
    assert np.all(left[inner] > idx[inner])
    kids = np.concatenate([left[inner], left[inner] + 1])
    assert np.array_equal(np.sort(kids), np.arange(1, t.size))     # every node but the root has one parent
    assert np.all(np.diff(left[inner]) == 2)                        # breadth first: children in parent order


def _hand_tree(thresholds):
    """A chain on feature 5: node 2k tests thresholds[k]; left child is a leaf of class 0, right goes on."""
    k = len(thresholds)
    n = 2 * k + 1
    left = -np.ones(n, np.int64)
    right = -np.ones(n, np.int64)
    feat = np.full(n, -2, np.int64)
    thr = np.full(n, -2.0)
    val = np.zeros((n, 2))
    node = 0
    for j, t in enumerate(thresholds):
        left[node], right[node] = node + 1, node + 2
        feat[node], thr[node] = 5, t
        val[node + 1] = (1.0, 0.0) if j % 2 == 0 else (0.0, 1.0)
        node += 2
    val[node] = (0.25, 0.75)
    return dict(children_left=left, children_right=right, feature=feat, threshold=thr, value=val,
                classes=np.array([0, 1], np.int64))


def test_round_down_thresholds(emul):
    # float64 thresholds exactly at, just above and just below float32 values, and between two of them
    f = np.float32(0.1)
    ts = [float(f), float(f) + 1e-12, float(f) - 1e-12, (float(f) + float(np.nextafter(f, np.float32(1)))) / 2,
          -1.5, float(np.finfo(np.float32).max), 1e300, np.inf, -np.inf, 0.0, -0.0, 1e-45, -1e-45]
    for t in ts:
        a = _hand_tree([t])
        vals = np.array([f, np.nextafter(f, np.float32(-1)), np.nextafter(f, np.float32(1)), -1.5, 0, -0.0, 1e-45,
                         -1e-45, np.finfo(np.float32).max, -np.finfo(np.float32).max, 3.0e38], np.float32)
        X = np.zeros((vals.size, 39), np.float32)
        X[:, 5] = vals
        labels, proba = emul_predict(emul, a, X)
        want = np.where(vals.astype(np.float64) <= t, 0, 1).astype(np.uint8)   # sklearn's float64 test
        assert np.array_equal(labels, want), t
        assert np.array_equal(ref_tree.speech(a, X), want)


def test_threshold_f32_is_round_down(emul):
    rng = np.random.default_rng(0)
    ts = np.concatenate([rng.normal(size=500) * 10 ** rng.uniform(-40, 38, 500), [3.4028235e38, 3.5e38]])
    a = _hand_tree(list(ts))
    rc, err, t, fl, leaves, depth = convert(emul, a)
    assert rc == 0, err
    inner = (fl >> 6) != np.arange(t.size)
    got = t[inner]
    # breadth first on a chain keeps the order of the tests
    for g, x in zip(got, ts):
        if x >= np.finfo(np.float32).max:
            assert np.isposinf(g)
            continue
        assert np.float64(g) <= x and (np.isneginf(g) or np.float64(np.nextafter(g, np.float32(np.inf))) > x)


def _malformed():
    good = _hand_tree([0.5, 1.0])
    cases = {}

    def case(name, **over):
        d = {k: np.array(v, copy=True) for k, v in good.items()}
        for k, v in over.items():
            d[k][...] = v
        cases[name] = d

    l, r = good["children_left"], good["children_right"]
    case("child out of range", children_right=np.where(np.arange(5) == 2, 9, r))
    case("child before parent", children_left=np.where(np.arange(5) == 2, 1, l))
    case("two parents", children_left=np.where(np.arange(5) == 2, 1, l), children_right=np.where(np.arange(5) == 2, 4, r))
    case("one child", children_right=np.where(np.arange(5) == 2, -1, r))
    case("feature out of range", feature=np.where(np.arange(5) == 0, 39, good["feature"]))
    case("negative feature", feature=np.where(np.arange(5) == 2, -2, good["feature"]))
    case("class 3", classes=[0, 3])
    case("negative class", classes=[-1, 1])
    case("classes not ascending", classes=[1, 0])
    case("NaN threshold", threshold=np.where(np.arange(5) == 0, np.nan, good["threshold"]))
    case("negative value", value=np.where(np.arange(10).reshape(5, 2) == 3, -1.0, good["value"]))
    case("NaN value", value=np.where(np.arange(10).reshape(5, 2) == 3, np.nan, good["value"]))
    cyc = {k: np.array(v, copy=True) for k, v in good.items()}
    cyc["children_left"][2], cyc["children_right"][2] = 0, 1        # a cycle back to the root
    cases["cycle"] = cyc
    return cases


@pytest.mark.parametrize("name", sorted(_malformed()))
def test_malformed_trees_are_rejected(emul, name):
    rc, err, *_ = convert(emul, _malformed()[name])
    assert rc == -1 and err


def test_unreachable_node_and_empty_tree_are_rejected(emul):
    a = _hand_tree([0.5])
    a = {k: (np.concatenate([v, v[-1:]]) if k != "classes" else v) for k, v in a.items()}
    rc, err, *_ = convert(emul, a)
    assert rc == -1 and "reachable" in err


def test_single_leaf_tree(emul):
    a = dict(children_left=np.array([-1]), children_right=np.array([-1]), feature=np.array([-2]),
             threshold=np.array([-2.0]), value=np.array([[0.2, 0.8]]), classes=np.array([0, 1]))
    a = {k: np.ascontiguousarray(v, dtype=np.float64 if k in ("threshold", "value") else np.int64) for k, v in a.items()}
    X = np.random.default_rng(1).normal(size=(10, 39)).astype(np.float32)
    labels, proba = emul_predict(emul, a, X)
    assert labels.all() and np.all(proba[:, 1] == np.float32(0.8))
    labels, _ = emul_predict(emul, a, X, 0.9)
    assert not labels.any()


def test_tree_arrays_sources(tmp_path):
    clf, X = fitted(2, max_depth=6)
    a = runtime.tree_arrays(clf)
    pk = tmp_path / "tree.pkl"
    with open(pk, "wb") as f:
        pickle.dump(clf, f)
    npz = tmp_path / "tree.npz"
    runtime.save_tree_npz(str(npz), clf)
    for src in (str(pk), str(npz), runtime.load_tree_npz(str(npz))):
        b = runtime.tree_arrays(src)
        assert all(np.array_equal(a[k], b[k]) for k in runtime.TREE_KEYS)
    counts = dict(a, value=a["value"] * 37.0)          # a tree that stores class counts (sklearn < 1.4)
    assert np.allclose(runtime.tree_arrays(counts)["value"], a["value"], rtol=1e-15, atol=0)
    with pytest.raises(ValueError):
        runtime.tree_arrays(dict(a, classes=np.array(["no", "yes"])))


def test_new_symbols_are_in_the_table():
    for name in ("vadb200_set_tree", "vadb200_clear_tree", "vadb200_get_classifier", "vadb200_tree_node_count",
                 "vadb200_tree_depth", "vadb200_tree_predict"):
        assert name in _lib.SIGNATURES
    so = os.path.join(ROOT, "vad_b200", "libvadb200.so")
    if os.path.isfile(so):
        lib = C.CDLL(so)
        for name in _lib.SIGNATURES:
            getattr(lib, name)
    hdr = open(os.path.join(ROOT, "include", "vadb200.h")).read()
    for name in ("vadb200_set_tree", "vadb200_tree_predict", "VADB200_CLASSIFIER_TREE"):
        assert name in hdr
