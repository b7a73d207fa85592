"""The training step's gradient and Adadelta update on the device, entry by entry against float64 (oracle/ref_train.py).

Reading the device gradient through the public API: a trainer with lr 2**16, rho 0, eps 2**40 takes one step from a
fresh optimizer state.  Its update kernel then computes a = g * g and, for |g| < 256, fl(a + eps) == 2**40, so
u = g * sqrtf(eps) / sqrtf(a + eps) == g bit for bit (IEEE sqrtf and division: the library is built without fast-math).
The new weight is p1 = fl(p0 - 2**16 g), and (p0 - p1) / 2**16 in float64 is g to within ulp(p1) / 2**17.

Tolerance of a gradient entry: |g_dev - g_ref| <= 1e-5 M + ulp(p1) / 2**17.  M is the backward pass of
ref_train.loss_and_grads on absolute values (|W|, activations, dlogits (p + y) / B; 0 for a clipped row), the a-priori
bound of the float32 sums, plus the first-order effect of the forward pass's own float32 error, taken as 1e-6 of each
value's absolute-value scale S_i = S_{i-1} |W_i| + |b_i|: an activation error of 1e-6 S_i in every weight-gradient
product, and a logit error of 1e-6 S4 in the dlogits, 2 p (1 - p) 1e-6 S4 / B.  Cancellation makes those errors large
next to the values themselves: a ReLU input a little above zero, or the logits of the x3 weights, which lose up to
~1e-2 (S4 ~ 1e5).  Every batch is free of near-ties, so float32 and float64 take the same ReLU and clip branches.
"""
import numpy as np
import pytest

from oracle import ref_math as rm, ref_train as rt

RTOL = 1e-5                 # float32 sums of the forward and backward pass, relative to their absolute-value bound
FWD_RTOL = 1e-6             # float32 activations and logits, relative to their absolute-value scale S_i
COL_SCALE = np.array([1.0] * 13 + [3.0] * 13 + [30.0] * 13)   # per-group scales of test_tc_ffn_rows_vs_oracle
READ_LR, READ_EPS = 2.0 ** 16, 2.0 ** 40
B200_SMS = 148

# batch sizes as functions of the SM count S: sub-tile, tile edges, grid edges (one tile per CTA), > 2 tiles per CTA
N_SPECS = {"1": lambda s: 1, "2": lambda s: 2, "127": lambda s: 127, "128": lambda s: 128, "129": lambda s: 129,
           "128S-1": lambda s: 128 * s - 1, "128S": lambda s: 128 * s, "128S+1": lambda s: 128 * s + 1,
           "2*128S+17*128+37": lambda s: 2 * 128 * s + 17 * 128 + 37}


def _weights(scale):
    """glorot_ffn plus N(0, 0.1) biases (non-zero, so the padding rows of a ragged tile have non-zero activations),
    the whole set times ``scale``; float32, as the device holds them."""
    w = rm.glorot_ffn(7)
    rng = np.random.default_rng(8)
    for i in (1, 2, 3, 4):
        w["b%d" % i] = rng.normal(0.0, 0.1, w["b%d" % i].shape).astype(np.float32)
    return {k: (v * np.float32(scale)).astype(np.float32) for k, v in w.items()}


def _forward(w, x, y):
    """float64 forward of the oracle's network with the absolute-value scales: activations, ReLU masks,
    S_i = S_{i-1} |W_i| + |b_i| (the scale of layer i's pre-activations), the smallest |z| / S of each row,
    probabilities, log p_true, log(1 - p_true) and the row maximum of S4."""
    p = {k: np.asarray(v, dtype=np.float64) for k, v in w.items()}
    a = np.asarray(x, dtype=np.float64)
    s = np.abs(a)
    acts, scales, masks, tie = [a], [np.zeros_like(a)], [], np.full(a.shape[0], np.inf)   # the input is exact
    for i in (1, 2, 3):
        z = a @ p["W%d" % i] + p["b%d" % i]
        sc = s @ np.abs(p["W%d" % i]) + np.abs(p["b%d" % i])
        tie = np.minimum(tie, (np.abs(z) / sc).min(axis=1))
        m = z > 0.0
        a, s = z * m, sc * m
        acts.append(a)
        scales.append(s)
        masks.append(m)
    z = a @ p["W4"] + p["b4"]
    s4 = (s @ np.abs(p["W4"]) + np.abs(p["b4"])).max(axis=1)
    lse = np.logaddexp.reduce(z, axis=1)
    prob = np.exp(z - lse[:, None])
    rows = np.arange(len(y))
    log_py = z[rows, y] - lse
    others = np.where(np.eye(3, dtype=bool)[y], -np.inf, z)
    log_rest = np.logaddexp.reduce(others, axis=1) - lse
    return dict(p=p, acts=acts, scales=scales, masks=masks, tie=tie, prob=prob, log_py=log_py, log_rest=log_rest,
                s4=s4)


def _clipped(f):
    return (f["log_py"] < np.log(1e-7)) | (f["log_rest"] < np.log(1e-7))


def _bound(w, x, y):
    """M: the backward pass on absolute values (see the module docstring)."""
    f = _forward(w, x, y)
    b = len(y)
    pr, onehot = f["prob"], np.eye(3)[y]
    d = (pr + onehot + (FWD_RTOL / RTOL) * 2.0 * pr * (1.0 - pr) * f["s4"][:, None]) / b
    d[_clipped(f)] = 0.0
    m = {}
    for i in (4, 3, 2, 1):
        m["W%d" % i] = (np.abs(f["acts"][i - 1]) + (FWD_RTOL / RTOL) * f["scales"][i - 1]).T @ d
        m["b%d" % i] = d.sum(axis=0)
        if i > 1:
            d = (d @ np.abs(f["p"]["W%d" % i]).T) * f["masks"][i - 2]
    return m


def _worst(g, g_ref, m, p1):
    """max over every entry of |g - g_ref| / (RTOL M + ulp(p1) / 2**17): <= 1 passes."""
    read = {k: np.spacing(np.abs(p1[k])).astype(np.float64) / 2 ** 17 for k in rt.KEYS}
    return max(float(np.max(np.abs(g[k] - g_ref[k]) / (RTOL * m[k] + read[k]))) for k in rt.KEYS)


def _near_tie(f):
    """A ReLU input within 1e-4 of its scale, or p_true (or 1 - p_true) within 0.1 % of 1e-7, widened by what an
    a-priori logit error of 1e-5 S4 moves its logarithm: 2 (1 - p_true) 1e-5 S4 (or 2 p_true 1e-5 S4)."""
    py = np.exp(f["log_py"])
    edge = np.log(1e-7)
    return ((f["tie"] < 1e-4) | (np.abs(f["log_py"] - edge) < 1e-3 + 2.0 * (1.0 - py) * RTOL * f["s4"])
            | (np.abs(f["log_rest"] - edge) < 1e-3 + 2.0 * py * RTOL * f["s4"]))


def _batch(w, n, seed, single_class=None, n_sms=B200_SMS):
    """n rows of N(0, 1) x COL_SCALE, labels of all three classes (or one), every 17th row all-zero, rows clipped at
    both ends in tile 0, in a CTA's second tile (tile S) and in the ragged tail.  A clipped row is an ordinary row
    times 60 labelled with its least (low end) or most (high end) likely class.  Near-tie rows are redrawn; returns
    x (float32), y (uint8) and the number of redraws."""
    rng = np.random.default_rng(seed)
    y = np.full(n, single_class) if single_class is not None else rng.integers(0, 3, n)
    zero = np.arange(n) % 17 == 16
    special = {}
    if single_class is None and n >= 4:
        starts = [0] + [128 * n_sms] * (n > 128 * n_sms) + [n - n % 128] * (n > 128 and n % 128 > 0)
        for r0 in starts:
            rows = [r for r in (r0 + 1, r0 + 2, r0) if r < n][:2]
            for r, kind in zip(rows, ("low", "high")):
                special[r] = kind
                zero[r] = False
    x = np.zeros((n, 39))
    todo = np.flatnonzero(~zero)
    redraws = -len(todo)
    while len(todo):
        redraws += len(todo)
        x[todo] = rng.standard_normal((len(todo), 39)) * COL_SCALE
        for r in todo:
            if r in special:
                x[r] *= 60.0
                pr = _forward(w, x[r:r + 1], y[r:r + 1])["prob"][0]
                y[r] = pr.argmin() if special[r] == "low" else pr.argmax()
        x32 = x.astype(np.float32)
        f = _forward(w, x32, y)
        bad = _near_tie(f)
        assert not np.any(bad & zero), "an all-zero row is a near-tie for these weights"
        bad[list(special)] |= ~_clipped(f)[list(special)]      # rare: two logits of a scaled row stay close
        todo = np.flatnonzero(bad)
    return x32, y.astype(np.uint8), redraws


def _tile_grad(w, x, y, t):
    """Tile t's contribution to the gradient of the whole batch (rows scaled by 1 / n)."""
    n = len(y)
    sl = slice(128 * t, min(n, 128 * t + 128))
    _, g = rt.loss_and_grads(w, x[sl], y[sl])
    return {k: v * ((sl.stop - sl.start) / n) for k, v in g.items()}


def _readout_p1(w, g):
    """The weights the read-out step leaves for gradient g: fl32(p0 - 2**16 g)."""
    return {k: (w[k].astype(np.float64) - READ_LR * g[k]).astype(np.float32) for k in rt.KEYS}


@pytest.mark.parametrize("name", [k for k in N_SPECS if N_SPECS[k](B200_SMS) > 128])
def test_gradient_criterion_rejects_a_lost_or_doubled_tile(name):
    """CPU: the comparison above, applied to oracle gradients with one full 128-row tile left out or counted twice (tile 0,
    a CTA's second tile and the last full tile), rejects them.  The x1 weights only: with the x3 set almost every row is
    clipped and the rest carry the logit-conditioning term, so a tile's share is below what float32 resolves there."""
    w = _weights(1.0)
    n = N_SPECS[name](B200_SMS)
    x, y, _ = _batch(w, n, seed=n)
    _, g = rt.loss_and_grads(w, x, y)
    m = _bound(w, x, y)
    full = n // 128
    for t in sorted({0, min(B200_SMS, full - 1), full - 1}):
        gt = _tile_grad(w, x, y, t)
        for sign in (-1.0, 1.0):
            bad = {k: g[k] + sign * gt[k] for k in rt.KEYS}
            assert _worst(bad, g, m, _readout_p1(w, bad)) > 1.0, (n, t, sign)


# ---- GPU -------------------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def dev():
    import torch
    from vad_b200 import runtime
    from vad_b200.trainer import FFNTrainer
    h = runtime.Handle()
    s = torch.cuda.get_device_properties(h.device).multi_processor_count
    n_max = N_SPECS["2*128S+17*128+37"](s)
    rd = FFNTrainer(h, weights=_weights(1.0), max_batch=n_max, lr=READ_LR, rho=0.0, eps=READ_EPS)
    yield h, s, rd
    rd.close()


def _to_dev(h, x, y):
    import torch
    return torch.from_numpy(x).to(h.device), torch.from_numpy(y).to(h.device)


def _read_gradient(rd, w, dx, dy):
    """One step of the read-out trainer from ``w`` with a fresh optimizer state: (loss, g, p1)."""
    rd.set_weights(w)
    loss = rd.train_on_batch(dx, dy)
    p1 = rd.weights()
    g = {k: (w[k].astype(np.float64) - p1[k].astype(np.float64)) / READ_LR for k in rt.KEYS}
    assert max(float(np.abs(v).max()) for v in g.values()) < 255.0, "u == g needs |g| < 256"
    return loss, g, p1


CASES = [(name, scale, None) for scale in (1.0, 3.0) for name in N_SPECS] + [("128S+1", 1.0, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,scale,single_class", CASES)
def test_gradients_match_float64(dev, name, scale, single_class):
    h, s, rd = dev
    w = _weights(scale)
    n = N_SPECS[name](s)
    x, y, redraws = _batch(w, n, seed=int(scale) * 1000 + n, single_class=single_class, n_sms=s)
    assert redraws <= 0.3 * n + 5 and (n < 1000 or redraws > 0), redraws
    f = _forward(w, x, y.astype(np.int64))
    clipped = _clipped(f)
    loss, g, p1 = _read_gradient(rd, w, *_to_dev(h, x, y))
    ref_loss, g_ref = rt.loss_and_grads(w, x, y.astype(np.int64))
    worst = _worst(g, g_ref, _bound(w, x, y.astype(np.int64)), p1)
    assert worst <= 1.0, (n, scale, worst, int(clipped.sum()))
    # the loss: float32 sums of positive terms, plus the logit-conditioning term of the unclipped rows; a row clipped
    # at the high end adds -log(fl32(1 - 1e-7)) = -log(1 - 2**-23), as float32 Keras, not the oracle's -log(1 - 1e-7)
    pc = np.exp(np.clip(f["log_py"], np.log(1e-7), np.log1p(-1e-7)))
    high = np.count_nonzero(f["log_rest"] < np.log(1e-7))
    tol = (RTOL * abs(ref_loss) + np.sum(np.where(clipped, 0.0, 2.0 * (1.0 - pc) * FWD_RTOL * f["s4"])) / n
           + high * (np.log1p(-1e-7) - np.log1p(-2.0 ** -23)) / n)
    assert abs(loss - ref_loss) <= tol, (n, scale, loss, ref_loss)


@pytest.mark.gpu
def test_batch_size_outside_one_to_max_batch_raises(dev):
    import torch
    from vad_b200._lib import VadB200Error
    h, s, rd = dev
    x, y = _to_dev(h, *(_batch(_weights(1.0), 4, seed=3, n_sms=s)[:2]))
    with pytest.raises(VadB200Error):
        rd.train_on_batch(x[:0].contiguous(), y[:0].contiguous())
    big = torch.zeros((rd.max_batch + 1, 39), dtype=torch.float32, device=h.device)
    with pytest.raises(VadB200Error):
        rd.train_on_batch(big, torch.zeros(rd.max_batch + 1, dtype=torch.uint8, device=h.device))


@pytest.mark.gpu
@pytest.mark.parametrize("lr,rho,eps", [(1.0, 0.95, 1e-8), (0.5, 0.9, 1e-6)])
def test_adadelta_update_matches_float64(dev, lr, rho, eps):
    """20 steps on a batch larger than the grid.  Before each step the read-out trainer gives the exact device gradient
    at the trainer's weights; float64 Adadelta on a float64 (a, d) state applies it to those weights, and the trainer's
    step must land within 2 float32 ulps of p plus 1e-6 of the step (plus what the read-out's ulp(p1) / 2**17 moves
    u).  Halfway, set_weights(..., reset_optimizer=False) keeps a and d; later reset_optimizer=True clears them."""
    from vad_b200.trainer import FFNTrainer
    h, s, rd = dev
    w0 = _weights(1.0)
    n = N_SPECS["2*128S+17*128+37"](s) - 1000
    x, y, _ = _batch(w0, n, seed=41, n_sms=s)
    dx, dy = _to_dev(h, x, y)
    tr = FFNTrainer(h, weights=w0, max_batch=n, lr=lr, rho=rho, eps=eps)
    twin = FFNTrainer(h, weights=w0, max_batch=n, lr=lr, rho=rho, eps=eps)
    lr, rho, eps = (float(np.float32(v)) for v in (lr, rho, eps))      # the device's constants
    a = {k: np.zeros(w0[k].shape) for k in rt.KEYS}
    d = {k: np.zeros(w0[k].shape) for k in rt.KEYS}
    rng = np.random.default_rng(5)
    worst = worst_ulps = 0.0
    for step in range(20):
        if step == 10:     # new weights, optimizer state kept
            cur = tr.weights()
            tr.set_weights({k: (v * (1 + 0.01 * rng.standard_normal(v.shape))).astype(np.float32)
                            for k, v in cur.items()}, reset_optimizer=False)
        if step == 15:     # optimizer state cleared
            tr.set_weights(tr.weights(), reset_optimizer=True)
            a = {k: np.zeros_like(v) for k, v in a.items()}
            d = {k: np.zeros_like(v) for k, v in d.items()}
        p0 = tr.weights()
        _, g, rp1 = _read_gradient(rd, p0, dx, dy)
        tr.train_on_batch(dx, dy, want_loss=False)
        if step == 0:      # deterministic: a second trainer from the same weights lands on the same bits
            twin.train_on_batch(dx, dy, want_loss=False)
            tw = twin.weights()
            assert all(np.array_equal(tw[k], v) for k, v in tr.weights().items())
        p1 = tr.weights()
        for k in rt.KEYS:
            a[k] = rho * a[k] + (1.0 - rho) * g[k] ** 2
            gain = np.sqrt(d[k] + eps) / np.sqrt(a[k] + eps)
            u = g[k] * gain
            ref = p0[k].astype(np.float64) - lr * u
            d[k] = rho * d[k] + (1.0 - rho) * u ** 2
            ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
            read_err = lr * gain * np.spacing(np.abs(rp1[k])).astype(np.float64) / 2 ** 17
            dev_err = np.abs(p1[k].astype(np.float64) - ref)
            tol = 2.0 * ulp + 1e-6 * lr * np.abs(u) + read_err
            assert np.all(dev_err <= tol), (step, k, (dev_err / tol).max())
            worst = max(worst, float((dev_err / tol).max()))
            ulp_bound = 2.0 * ulp >= tol / 2          # entries whose tolerance is mostly the ulp term
            worst_ulps = max(worst_ulps, float((dev_err / ulp)[ulp_bound].max(initial=0.0)))
    print("adadelta lr=%g rho=%g eps=%g: worst deviation / tolerance %.3f, %.3f float32 ulps where ulps bound it"
          % (lr, rho, eps, worst, worst_ulps))
    tr.close()
    twin.close()
