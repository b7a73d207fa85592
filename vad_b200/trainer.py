"""Classifier training on the device: drop-ins for learning/ffn_trainer.py:104-175 (``FFNTrainer``, ``train``) and
learning/decision_classifier_trainer.py (``fit_tree``).

``FFNTrainer.train_on_batch(x, y)`` is Keras-1 ``model.train_on_batch`` for the reference's network and compile
settings (categorical cross-entropy, Adadelta lr 1.0 / rho 0.95 / eps 1e-8) as two CUDA kernels per step
(``vadb200_train_on_batch``).  Features are the rows the fused kernels produce (``batch.process_files`` /
``FeatureStore``), so the feature kernel is the data loader; ``mixing_batches`` restates the class-mixing generator of
dataset/__init__.py:38-96 as index arithmetic on device-resident per-class row tensors.  Weights round-trip through the
``.npz`` container of ``runtime.load_ffn_npz`` into ``Handle.set_ffn_weights`` (model.save_weights / load_weights).
"""
import ctypes as C

import numpy as np
import torch

from . import runtime
from ._lib import check
from .runtime import FFN_KEYS, FFN_SHAPES

ACCURACY_THRESHOLD = 0.90       # ffn_trainer.py:22
BATCH_SIZE = 32                 # ffn_trainer.py:15 (the device step is built for batches of thousands)
EPOCHS_NUM = 25                 # ffn_trainer.py:16


def mixing_batches(sizes, batch_size, rng):
    """dataset/__init__.py:38-96: the order in which samples of the class sources are drawn (stochastic roulette over
    the remaining sizes, without replacement), cut into batches.  Yields int64 arrays of source indices."""
    remaining = [int(s) for s in sizes]
    total = sum(remaining)
    buf = []
    drawn = 0
    while drawn < total:
        tb = float(sum(remaining))
        w = [r / tb for r in remaining]
        idx = rng.randint(len(remaining))
        mw = max(w)
        b = 0.0
        for _ in range(len(remaining)):
            if drawn == total:
                break
            b += rng.random() * 2 * mw
            while w[idx] <= b:
                b -= w[idx]
                idx = 0 if idx == len(remaining) - 1 else idx + 1
            if remaining[idx] == 0:
                return
            remaining[idx] -= 1
            drawn += 1
            buf.append(idx)
            if len(buf) == batch_size:
                yield np.asarray(buf, dtype=np.int64)
                buf = []


class FFNTrainer(object):
    def __init__(self, handle=None, weights=None, seed=0, max_batch=4096, lr=1.0, rho=0.95, eps=1e-8):
        self.handle = handle or runtime.Handle()
        self.lib = self.handle.lib
        self.max_batch = int(max_batch)
        self._t = C.c_void_p()
        check(self.lib.vadb200_trainer_create(self.handle._h, self.max_batch, lr, rho, eps, C.byref(self._t)))
        self.set_weights(weights if weights is not None else runtime.glorot_ffn(seed))   # Keras-1 Dense default init

    def close(self):
        if getattr(self, "_t", None) is not None and self._t:
            self.lib.vadb200_trainer_destroy(self._t)
            self._t = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_weights(self, w, reset_optimizer=True):
        arrs = [np.ascontiguousarray(np.asarray(w[k], dtype=np.float32)) for k in FFN_KEYS]
        for k, a in zip(FFN_KEYS, arrs):
            if a.shape != FFN_SHAPES[k]:
                raise ValueError("FFN weight %s must have shape %r, got %r" % (k, FFN_SHAPES[k], a.shape))
        check(self.lib.vadb200_trainer_set_weights(self._t, *[a.ctypes.data_as(C.c_void_p) for a in arrs],
                                                   1 if reset_optimizer else 0))

    def weights(self):
        out = {k: np.empty(FFN_SHAPES[k], dtype=np.float32) for k in FFN_KEYS}
        check(self.lib.vadb200_trainer_get_weights(self._t, *[out[k].ctypes.data_as(C.c_void_p) for k in FFN_KEYS]))
        return out

    def train_on_batch(self, x, y, want_loss=True):
        """x: [n, 39] float32 CUDA tensor, y: [n] uint8 CUDA tensor of class ids.  Returns the batch loss (computed
        before the update, as Keras) or None."""
        if not (torch.is_tensor(x) and x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 2
                and x.shape[1] == 39):
            raise TypeError("x must be a contiguous [n, 39] float32 CUDA tensor")
        if not (torch.is_tensor(y) and y.is_cuda and y.dtype == torch.uint8 and y.is_contiguous()
                and y.shape == (x.shape[0],)):
            raise TypeError("y must be a contiguous [n] uint8 CUDA tensor")
        loss = C.c_float()
        check(self.lib.vadb200_train_on_batch(self._t, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), x.shape[0],
                                              C.byref(loss) if want_loss else None, self.handle.stream))
        return loss.value if want_loss else None

    def sync_classifier(self):
        """Install the current weights in the handle (model.load_weights into the inference path)."""
        self.handle.set_ffn_weights(self.weights())

    def evaluate(self, x, y):
        """model.evaluate: (mean categorical cross-entropy, accuracy over the three classes) with the inference path."""
        self.sync_classifier()
        _, logits = self.handle.ffn_predict(x)
        lg = logits.double()
        logp = lg - torch.logsumexp(lg, dim=1, keepdim=True)
        pc = logp.gather(1, y.long()[:, None]).exp().clamp(1e-7, 1 - 1e-7)
        return float(-pc.log().mean()), float((lg.argmax(dim=1) == y.long()).double().mean())

    def save(self, path):
        """model.save_weights (ffn_trainer.py:165,175) as the .npz container ``runtime.load_ffn_npz`` reads."""
        np.savez(path, **self.weights())


def train(trainer, sources, epochs=EPOCHS_NUM, batch_size=4096, val_fraction=0.25, seed=0, save_prefix=None, log=print):
    """The epoch loop of ffn_trainer.py:127-175.  ``sources``: list of (rows [n_c, 39] float32 CUDA tensor, class id),
    e.g. noise (0), speech (1), music (2).  Each epoch draws mixed batches (dataset/__init__.py:38-96) from the training
    part of every source, calls train_on_batch, then evaluates on the held-out part; weights are saved when validation
    accuracy first exceeds ACCURACY_THRESHOLD and at the end."""
    rng = np.random.RandomState(seed)
    train_parts, val_x, val_y = [], [], []
    for rows, cls in sources:
        n_val = int(rows.shape[0] * val_fraction)
        train_parts.append((rows[n_val:], cls))
        val_x.append(rows[:n_val])
        val_y.append(torch.full((n_val,), cls, dtype=torch.uint8, device=rows.device))
    val_x, val_y = torch.cat(val_x).contiguous(), torch.cat(val_y)
    model_ready = False
    history = []
    for epoch in range(epochs):
        cursors = [torch.randperm(p.shape[0], device=p.device) for p, _ in train_parts]   # random line access
        used = [0] * len(train_parts)
        for src in mixing_batches([p.shape[0] for p, _ in train_parts], batch_size, rng):
            xs, ys = [], []
            for c, (rows, cls) in enumerate(train_parts):
                k = int((src == c).sum())
                if k:
                    xs.append(rows[cursors[c][used[c]:used[c] + k]])
                    ys.append(torch.full((k,), cls, dtype=torch.uint8, device=rows.device))
                    used[c] += k
            trainer.train_on_batch(torch.cat(xs).contiguous(), torch.cat(ys), want_loss=False)
        val_loss, val_acc = trainer.evaluate(val_x, val_y)
        history.append((val_loss, val_acc))
        if log:
            log("Epoch %d  validation score %.5f  accuracy %.4f" % (epoch, val_loss, val_acc))
        if val_acc > ACCURACY_THRESHOLD and not model_ready:
            if save_prefix:
                trainer.save(save_prefix + "_achieved_accuracy.npz")
            model_ready = True
    if save_prefix:
        trainer.save(save_prefix + "_full_training.npz")
    return history


# learning/decision_classifier_trainer.py's grid-search best (cross_validation.res)
TREE_MAX_DEPTH = 25
TREE_MIN_SAMPLES_LEAF = 20
TREE_MIN_SAMPLES_SPLIT = 22


def fit_tree(sources, val_fraction=0.25, max_depth=TREE_MAX_DEPTH, min_samples_leaf=TREE_MIN_SAMPLES_LEAF,
             min_samples_split=TREE_MIN_SAMPLES_SPLIT, seed=0, save_path=None, handle=None, log=print):
    """The flow of learning/decision_classifier_trainer.py on the device.  ``sources``: list of (rows [n_c, 39] float32
    CUDA tensor, class id).  Rows with a non-finite feature are dropped (and counted in the log); a random
    ``val_fraction`` of each source is held out; the tree is fitted on the rest (``runtime.TreeFitter``) and scored on
    the held-out rows with ``Handle.tree_predict`` (clf.score: the class of the largest probability equals the label).
    ``save_path``: the tree's arrays go to an .npz (``runtime.save_tree_npz``; replaces cPickle.dump).
    Returns (tree dict, held-out accuracy; NaN without held-out rows)."""
    handle = handle or runtime.Handle()
    g = torch.Generator(device="cpu").manual_seed(int(seed))
    fit_x, fit_y, val_x, val_y = [], [], [], []
    for rows, cls in sources:
        ok = torch.isfinite(rows).all(dim=1)
        dropped = int((~ok).sum())
        if dropped and log:
            log("class %d: dropped %d rows with a non-finite feature" % (cls, dropped))
        rows = rows[ok]
        perm = torch.randperm(rows.shape[0], generator=g).to(rows.device)
        n_val = int(rows.shape[0] * val_fraction)
        for xs, ys, part in ((val_x, val_y, perm[:n_val]), (fit_x, fit_y, perm[n_val:])):
            xs.append(rows[part])
            ys.append(torch.full((part.shape[0],), cls, dtype=torch.uint8, device=rows.device))
    x, y = torch.cat(fit_x).contiguous(), torch.cat(fit_y).contiguous()
    fitter = runtime.TreeFitter(handle, x.shape[0])
    try:
        tree = fitter.fit(x, y, max_depth=max_depth, min_samples_split=min_samples_split,
                          min_samples_leaf=min_samples_leaf)
    finally:
        fitter.close()
    vx, vy = torch.cat(val_x).contiguous(), torch.cat(val_y)
    accuracy = float("nan")
    if vx.shape[0]:
        scorer = runtime.Handle(handle.device)
        try:
            scorer.set_tree(tree)
            _, proba = scorer.tree_predict(vx)
            accuracy = float((proba.argmax(dim=1) == vy.long()).double().mean())
        finally:
            scorer.close()
    if log:
        log("tree: %d nodes, %d tied, fitted on %d rows, held-out accuracy %.4f"
            % (tree["feature"].shape[0], tree["tied_nodes"], x.shape[0], accuracy))
    if save_path:
        runtime.save_tree_npz(save_path, tree)
    return tree, accuracy
