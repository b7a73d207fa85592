"""CPU restatement of one optimisation step of the reference's FFN trainer (TEST INFRASTRUCTURE; parity unpinned).

learning/ffn_trainer.py:104-120 builds Sequential(Dense64 relu relu Dense32 relu Dense16 relu Dense3 softmax) and
compiles it with loss='categorical_crossentropy', optimizer='adadelta'; :148 calls model.train_on_batch.  Keras 1.x
is neither vendored nor installed, so its arithmetic is restated from its published source (keras/objectives.py,
keras/optimizers.py of the 1.x line): softmax output clipped to [1e-7, 1 - 1e-7] inside the cross-entropy, mean over
the batch.  The clip's gradient (Theano T.clip, TF clip_by_value) is zero outside that closed interval, so a row whose
unclipped true-class probability lies outside it adds its clipped value to the loss and nothing to the gradient.
Adadelta(lr=1.0, rho=0.95, epsilon=1e-8):
    a <- rho a + (1 - rho) g^2;  u = g sqrt(d + eps) / sqrt(a + eps);  p <- p - lr u;  d <- rho d + (1 - rho) u^2
All in float64.  ``mixing_order`` restates the class-mixing generator of dataset/__init__.py:38-96.
"""
import numpy as np

KEYS = ("W1", "b1", "W2", "b2", "W3", "b3", "W4", "b4")


def init_state(w):
    p = {k: np.asarray(w[k], dtype=np.float64).copy() for k in KEYS}
    return {"p": p, "a": {k: np.zeros_like(v) for k, v in p.items()}, "d": {k: np.zeros_like(v) for k, v in p.items()}}


def loss_and_grads(p, x, y):
    """x [B, 39], y [B] class ids -> (loss, grads dict).  ffn_trainer.py:106-116 forward, exact backward."""
    x = np.asarray(x, dtype=np.float64)
    b = x.shape[0]
    acts = [x]
    h = x
    for i in (1, 2, 3):
        h = np.maximum(h @ p["W%d" % i] + p["b%d" % i], 0.0)
        acts.append(h)
    logits = h @ p["W4"] + p["b4"]
    z = logits - logits.max(axis=1, keepdims=True)
    e = np.exp(z)
    prob = e / e.sum(axis=1, keepdims=True)
    onehot = np.eye(3)[np.asarray(y, dtype=np.int64)]
    py = (prob * onehot).sum(axis=1)
    loss = float(-np.log(np.clip(py, 1e-7, 1.0 - 1e-7)).mean())
    live = (py >= 1e-7) & (py <= 1.0 - 1e-7)        # the clip passes a gradient on the closed interval only
    d = (prob - onehot) * (live[:, None] / b)
    g = {}
    for i in (4, 3, 2, 1):
        a_prev = acts[i - 1]
        g["W%d" % i] = a_prev.T @ d
        g["b%d" % i] = d.sum(axis=0)
        if i > 1:
            d = (d @ p["W%d" % i].T) * (a_prev > 0.0)
    return loss, g


def train_on_batch(state, x, y, lr=1.0, rho=0.95, eps=1e-8):
    """One Keras-1 ``train_on_batch``: returns the loss computed BEFORE the update, updates ``state`` in place."""
    loss, g = loss_and_grads(state["p"], x, y)
    for k in KEYS:
        a = rho * state["a"][k] + (1.0 - rho) * g[k] ** 2
        u = g[k] * np.sqrt(state["d"][k] + eps) / np.sqrt(a + eps)
        state["p"][k] = state["p"][k] - lr * u
        state["a"][k] = a
        state["d"][k] = rho * state["d"][k] + (1.0 - rho) * u ** 2
    return loss


def mixing_order(sizes, rng):
    """dataset/__init__.py:38-96 ``random_features_generator`` as a sequence of source indices: a stochastic roulette
    over the sources weighted by their REMAINING sizes, without replacement; yields up to sum(sizes) indices (the
    reference ends early if a source runs dry between two refreshes of the weights).  ``rng`` needs
    ``randint(n)`` and ``random()`` (np.random.RandomState, as the reference's module-level np.random)."""
    remaining = [int(s) for s in sizes]
    total = sum(remaining)
    out = []
    while len(out) < total:
        tb = float(sum(remaining))
        w = [r / tb for r in remaining]
        idx = rng.randint(len(remaining))
        mw = max(w)
        b = 0.0
        for _ in range(len(remaining)):
            if len(out) == total:
                break
            b += rng.random() * 2 * mw
            while w[idx] <= b:
                b -= w[idx]
                idx = 0 if idx == len(remaining) - 1 else idx + 1
            if remaining[idx] == 0:        # :86-91: the exhausted source raises StopIteration, which ends this generator
                return np.asarray(out, dtype=np.int64)   # too (the weights w are only refreshed every len(sizes) draws)
            remaining[idx] -= 1
            out.append(idx)
    return np.asarray(out, dtype=np.int64)
