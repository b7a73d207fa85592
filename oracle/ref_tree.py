"""sklearn DecisionTreeClassifier's apply / predict / predict_proba (sklearn 1.9, single output) restated in numpy:
X is cast to float32 and each node compares float64(x) <= threshold; predict is classes_[argmax(value[leaf])] (the
first maximum), predict_proba is value[leaf] as stored (class fractions).  ``t`` is a dict of the arrays
vadb200_set_tree takes (vad_b200.runtime.tree_arrays)."""
import numpy as np


def apply(t, X):
    X = np.asarray(X, dtype=np.float32)
    left, right = np.asarray(t["children_left"]), np.asarray(t["children_right"])
    feat, thr = np.asarray(t["feature"]), np.asarray(t["threshold"], dtype=np.float64)
    node = np.zeros(X.shape[0], dtype=np.int64)
    rows = np.arange(X.shape[0])
    while True:
        inner = left[node] != -1
        if not inner.any():
            return node
        r, n = rows[inner], node[inner]
        go_left = X[r, feat[n]].astype(np.float64) <= thr[n]
        node[inner] = np.where(go_left, left[n], right[n])


def predict_proba(t, X):
    return np.asarray(t["value"], dtype=np.float64)[apply(t, X)]


def predict(t, X):
    return np.asarray(t["classes"])[np.argmax(predict_proba(t, X), axis=1)]


def speech(t, X, threshold=0.0):
    """The library's decision: predict == 1 (threshold <= 0) or predict_proba's class-1 column >= threshold."""
    cls = list(np.asarray(t["classes"]))
    if threshold <= 0:
        return (predict(t, X) == 1).astype(np.uint8)
    if 1 not in cls:
        return np.zeros(np.asarray(X).shape[0], np.uint8)
    return (predict_proba(t, X)[:, cls.index(1)] >= np.float64(np.float32(threshold))).astype(np.uint8)


def proba_by_id(t, X):
    """float32 probabilities in the columns of class ids 0, 1, 2 (0 for a class the tree lacks)."""
    p = predict_proba(t, X)
    out = np.zeros((p.shape[0], 3), np.float32)
    for k, c in enumerate(np.asarray(t["classes"])):
        out[:, int(c)] = p[:, k].astype(np.float32)
    return out
