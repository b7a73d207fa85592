"""Decision-tree fit without a GPU: tests/_ref_tree_fit.py (the restatement vadb200_tree_fit is held to) against
sklearn 1.9 on specs chosen to be tie-free, an independent brute-force certificate of its choices on specs with ties,
and the lowest-feature tie rule."""
import numpy as np
import pytest

import _ref_tree_fit as R

sklearn_tree = pytest.importorskip("sklearn.tree")

REF = dict(max_depth=25, min_samples_leaf=20, min_samples_split=22)


def _rules(X):
    """Axis-aligned, noise-free labels: every impure node has one clearly best split."""
    y = (X[:, 0] > 0.1).astype(np.int64)
    y[X[:, 3] > 0.9] = 2
    y[X[:, 7] < -1.2] = 0
    y[(X[:, 12] > 1.0) & (X[:, 0] > 0.1)] = 0
    return y


def _band(rng, n, lo, step, ulps):
    """Values on a grid of `step` from `lo`, each moved by up to `ulps` float32 ulps (near-equal neighbours)."""
    base = (lo + step * rng.integers(0, 64, n)).astype(np.float32)
    for _ in range(ulps):
        up = rng.random(n) < 0.5
        base = np.where(up, np.nextafter(base, np.float32(np.inf)), base).astype(np.float32)
    return base


# Data seeds under which each spec is tie-free (a stray row that min_samples_leaf keeps from its own leaf lets many
# features reach the same proxy, so not every seed is).
SEEDS = {"ref": 3, "unbounded": 1}


def spec(name, seed=None):
    """(X [n, 39] float32, y int64, fit kwargs) of each named case."""
    rng = np.random.default_rng(SEEDS.get(name, 0) if seed is None else seed)
    n = 6000
    X = rng.normal(size=(n, 39)).astype(np.float32)
    y = _rules(X)
    kw = {}
    if name == "stump":
        kw = dict(max_depth=1)
    elif name == "depth3":
        kw = dict(max_depth=3)
    elif name == "ref":
        kw = dict(REF)
    elif name == "unbounded":
        kw = dict(min_samples_leaf=5)
    elif name == "classes02":
        y = np.where(y == 1, 2, 0)
        kw = dict(max_depth=4)
    elif name == "single":
        y = np.full(n, 1)
    elif name == "tiny":
        X, y, kw = X[:15], y[:15], dict(REF)
    elif name == "constant":
        X[:, 0] = 1.5
        X[:, 5] = -3.0
        kw = dict(max_depth=4)
    elif name == "decrease":
        kw = dict(min_impurity_decrease=0.01)
    elif name in ("band1", "band1k", "bandtiny"):
        lo, step = {"band1": (1.0, 1.0 / 64), "band1k": (1024.0, 8.0), "bandtiny": (1e-5, 1e-5)}[name]
        for f in (0, 3, 7, 12):
            X[:, f] = _band(rng, n, lo, step, 3)
        y = _rules((X - lo) / (64 * step) * 4 - 2)
        kw = dict(max_depth=3)
    return np.ascontiguousarray(X), y, kw


TIE_FREE = ["stump", "depth3", "ref", "unbounded", "classes02", "single", "tiny", "constant", "decrease", "band1",
            "band1k", "bandtiny"]


@pytest.mark.parametrize("name", TIE_FREE)
def test_oracle_equals_sklearn(name):
    X, y, kw = spec(name)
    t = R.fit(X, y, **kw)
    assert t["tied_nodes"] == 0, "spec %s must be tie-free" % name
    for rs in (0, 1, 2):
        clf = sklearn_tree.DecisionTreeClassifier(random_state=rs, **kw).fit(X, y)
        assert R.same_tree(t, R.sklearn_arrays(clf)), "random_state %d" % rs
    if name in ("single", "tiny"):
        assert t["feature"].shape == (1,)


def test_specs_cover_their_cases():
    assert list(spec("classes02")[1].tolist().count(c) > 0 for c in (0, 1, 2)) == [True, False, True]
    assert len(R.fit(*spec("ref")[:2], **spec("ref")[2])["feature"]) >= 15
    assert spec("tiny")[0].shape[0] < REF["min_samples_split"]
    X, y, kw = spec("decrease")
    assert len(R.fit(X, y, **kw)["feature"]) < len(R.fit(X, y)["feature"])
    X = spec("band1")[0][:, 0]
    assert np.all((X >= 1) & (X < 2))
    srt = np.unique(X)
    assert np.any(np.diff(srt) > 0) and np.any(srt[1:] <= srt[:-1] + np.float32(1e-7))   # one-ulp neighbours merge
    X = spec("bandtiny")[0][:, 0]
    srt = np.unique(X)
    assert np.any(srt[1:] <= srt[:-1] + np.float32(1e-7))                                   # chains below 1e-3


def certify(X, y, t, min_samples_leaf=1, min_samples_split=2, max_depth=None, min_impurity_decrease=0.0):
    """Brute force, O(m^2) per node and feature: every internal node takes the maximum proxy, the lowest feature among
    the maxima and the earliest position; every leaf meets a stopping rule or has no candidate."""
    X = np.asarray(X, np.float32)
    mss = max(min_samples_split, 2 * min_samples_leaf)
    rows = {0: np.arange(X.shape[0])}
    depth = {0: 0}
    for k in range(t["feature"].shape[0]):
        r = rows[k]
        m = r.shape[0]
        assert t["n_node_samples"][k] == m
        best = None
        for f in range(39):
            v = np.sort(X[r, f], kind="stable")
            for p in range(1, m):
                if not (v[p] > np.float32(v[p - 1] + np.float32(1e-7))):
                    continue
                if p < min_samples_leaf or m - p < min_samples_leaf:
                    continue
                go = X[r, f] < v[p]
                cl = np.bincount(y[r][go], minlength=3)
                cr = np.bincount(y[r][~go], minlength=3)
                px = -(float(m - p) * float(R.gini(cr, m - p))) - (float(p) * float(R.gini(cl, p)))
                if best is None or px > best[0]:
                    best = (px, f, p, float(np.float64(v[p - 1]) / 2.0 + np.float64(v[p]) / 2.0))
        leaf = t["children_left"][k] == -1
        stop = (max_depth is not None and depth[k] >= max_depth) or m < mss or t["impurity"][k] <= R.EPSILON
        if leaf:
            assert stop or best is None or min_impurity_decrease > 0, "leaf %d has a split" % k
            continue
        assert best is not None and not stop
        assert (t["feature"][k], t["threshold"][k]) == (best[1], best[3]), "node %d" % k
        go = X[r, best[1]].astype(np.float64) <= t["threshold"][k]
        rows[t["children_left"][k]], rows[t["children_right"][k]] = r[go], r[~go]
        depth[t["children_left"][k]] = depth[t["children_right"][k]] = depth[k] + 1


@pytest.mark.parametrize("seed", [0, 1])
def test_certificate_on_specs_with_ties(seed):
    rng = np.random.default_rng(seed)
    n = 400
    X = rng.normal(size=(n, 39)).astype(np.float32)
    y = ((X[:, :3].sum(axis=1) + rng.normal(size=n)) > 0).astype(np.int64)
    y[rng.random(n) < 0.1] = 2
    kw = dict(min_samples_leaf=5)
    t = R.fit(X, y, **kw)
    assert t["tied_nodes"] > 0
    certify(X, y, t, **kw)


def test_identical_columns_split_on_the_lower_index():
    rng = np.random.default_rng(5)
    n = 2000
    X = rng.normal(size=(n, 39)).astype(np.float32)
    X[:, 30] = X[:, 11]
    y = (X[:, 11] > 0.3).astype(np.int64)
    t = R.fit(X, y, max_depth=1)
    assert t["feature"][0] == 11 and t["tied_nodes"] == 1
    picks = {int(sklearn_tree.DecisionTreeClassifier(max_depth=1, random_state=rs).fit(X, y).tree_.feature[0])
             for rs in range(12)}
    assert picks == {11, 30}
