"""The Gini decision-tree fit of vadb200_tree_fit restated in plain numpy float64: sklearn 1.9's
DecisionTreeClassifier(criterion="gini", splitter="best", max_features=None) built node by node in depth-first
preorder (left child first), except that among features reaching the same best proxy the lowest index wins.
``tied_nodes`` counts the nodes where that rule decided, so tied_nodes == 0 means sklearn builds this tree for every
random_state.

Per node: sort the node's rows by each feature; position p is a candidate iff x[p] > x[p-1] + 1e-7 in float32 and
both sides keep min_samples_leaf rows; proxy = -(n_r g_r) - (n_l g_l) with g = 1.0 - sum(count^2) / (n n) in float64;
within a feature the first maximum wins; threshold = double(x[p-1]) / 2.0 + double(x[p]) / 2.0.  Returns the dict
``runtime.tree_arrays`` accepts plus impurity, n_node_samples and tied_nodes."""
import numpy as np

FEATURE_THRESHOLD = np.float32(1e-7)
EPSILON = float(np.finfo(np.float64).eps)
_BLOCK = 1 << 22   # rows x features per vectorised block


def gini(counts, n):
    """1.0 - sum(count^2) / (n n), summed class by class as sklearn's Gini does."""
    c = np.asarray(counts, dtype=np.float64)
    w = np.asarray(n, dtype=np.float64)
    sq = c[..., 0] * c[..., 0] + c[..., 1] * c[..., 1] + c[..., 2] * c[..., 2]
    return 1.0 - sq / (w * w)


def best_split(X, y, min_samples_leaf):
    """(feature, position, threshold, tie, best proxy) of the node with rows X [m, F] float32 / y [m], or None."""
    m, F = X.shape
    tot = np.bincount(y, minlength=3)
    per = np.full(F, -np.inf)
    pos = np.zeros(F, dtype=np.int64)
    orders = {}
    step = max(1, _BLOCK // max(m, 1))
    p = np.arange(1, m, dtype=np.int64)
    nl, nr = p, m - p
    ok_n = (nl >= min_samples_leaf) & (nr >= min_samples_leaf)
    for f0 in range(0, F, step):
        fs = slice(f0, min(F, f0 + step))
        order = np.argsort(X[:, fs], axis=0, kind="stable")
        xs = np.take_along_axis(X[:, fs], order, axis=0)
        onehot = np.eye(3, dtype=np.int64)[y[order]]                  # [m, f, 3]
        left = np.cumsum(onehot, axis=0)[:-1]                          # counts at positions < p, p = 1 .. m-1
        cand = (xs[1:] > (xs[:-1] + FEATURE_THRESHOLD)) & ok_n[:, None]
        gl = gini(left, nl[:, None])
        gr = gini(tot - left, nr[:, None])
        proxy = -(nr[:, None] * gr) - (nl[:, None] * gl)
        proxy = np.where(cand, proxy, -np.inf)
        if proxy.shape[0] == 0:
            continue
        idx = np.argmax(proxy, axis=0)
        per[fs] = proxy[idx, np.arange(proxy.shape[1])]
        pos[fs] = idx + 1
        for j in range(fs.stop - fs.start):
            orders[f0 + j] = (order[:, j], xs[:, j])
    best = per.max() if F else -np.inf
    if best == -np.inf:
        return None
    ties = np.flatnonzero(per == best)
    f = int(ties[0])
    order, xs = orders[f]
    q = int(pos[f])
    thr = float(np.float64(xs[q - 1]) / 2.0 + np.float64(xs[q]) / 2.0)
    return f, q, thr, len(ties) > 1, float(best), order


def fit(X, y, max_depth=None, min_samples_split=2, min_samples_leaf=1, min_impurity_decrease=0.0):
    X = np.ascontiguousarray(X, dtype=np.float32)
    y = np.asarray(y).astype(np.int64)
    n = y.shape[0]
    classes = np.unique(y)
    mss = max(int(min_samples_split), 2 * int(min_samples_leaf))
    md = max_depth if (max_depth is not None and max_depth > 0) else np.inf
    L, R, FE, TH, IMP, NS, CNT = [], [], [], [], [], [], []
    tied = 0
    stack = [(np.arange(n), 0, -1, False)]
    while stack:
        rows, depth, parent, is_left = stack.pop()
        node = len(L)
        if parent >= 0:
            (L if is_left else R)[parent] = node
        m = rows.shape[0]
        cnt = np.bincount(y[rows], minlength=3)
        imp = float(gini(cnt, m))
        L.append(-1), R.append(-1), FE.append(-2), TH.append(-2.0), IMP.append(imp), NS.append(m), CNT.append(cnt)
        if depth >= md or m < mss or m < 2 * min_samples_leaf or imp <= EPSILON:
            continue
        s = best_split(X[rows], y[rows], min_samples_leaf)
        if s is None:
            continue
        f, q, thr, tie, _, order = s
        tied += int(tie)
        lrows, rrows = rows[order[:q]], rows[order[q:]]
        cl, cr = np.bincount(y[lrows], minlength=3), np.bincount(y[rrows], minlength=3)
        wn, wl, wr = float(m), float(q), float(m - q)
        il, ir = float(gini(cl, q)), float(gini(cr, m - q))
        improvement = (wn / n) * (imp - (wr / wn) * ir - (wl / wn) * il)
        if improvement + EPSILON < min_impurity_decrease:
            continue
        FE[node], TH[node] = f, thr
        stack.append((rrows, depth + 1, node, False))
        stack.append((lrows, depth + 1, node, True))
    cnt = np.asarray(CNT, dtype=np.float64)
    ns = np.asarray(NS, dtype=np.int64)
    return dict(children_left=np.asarray(L, np.int64), children_right=np.asarray(R, np.int64),
                feature=np.asarray(FE, np.int64), threshold=np.asarray(TH, np.float64),
                value=cnt[:, classes] / ns[:, None].astype(np.float64), impurity=np.asarray(IMP, np.float64),
                n_node_samples=ns, classes=classes.astype(np.int64), tied_nodes=int(tied))


ARRAYS = ("children_left", "children_right", "feature", "threshold", "value", "impurity", "n_node_samples", "classes")


def sklearn_arrays(clf):
    """The same dict from a fitted sklearn DecisionTreeClassifier."""
    t = clf.tree_
    return dict(children_left=t.children_left, children_right=t.children_right, feature=t.feature,
                threshold=t.threshold, value=np.asarray(t.value)[:, 0, :], impurity=t.impurity,
                n_node_samples=t.n_node_samples, classes=np.asarray(clf.classes_, dtype=np.int64))


def same_tree(a, b):
    """Array for array, bit for bit."""
    return all(_bits(a[k]).shape == _bits(b[k]).shape and np.array_equal(_bits(a[k]), _bits(b[k])) for k in ARRAYS)


def _bits(v):
    v = np.asarray(v)
    return np.ascontiguousarray(v, dtype=np.float64).view(np.int64) if v.dtype.kind == "f" else v.astype(np.int64)
