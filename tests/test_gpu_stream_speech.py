"""GPU: speech segments on the stream bank (vadb200_stream_bank_set_speech / _feed_speech / _end_streams).  Each
stream's finalised rows, with the tail its end resolves, equal oracle/ref_segments.py over the stream's own labels;
for whole utterances they equal batch.speech_segments; ending streams leaves the others byte-identical; labels and
logits do not change when speech is on."""
import numpy as np
import pytest

from oracle import ref_math as rm, ref_segments as rs
from vad_b200.synth import synth_utterance

import _signals
from test_gpu_segments import GRID

pytestmark = pytest.mark.gpu

WARM = 7


def delay(S, G, P):
    return (G - 1 if G > 1 else 0) + (S - 1 if S > 1 else 0) + P


def gated_weights():
    """A classifier that says speech for every row with finite features: rows whose five frames are digital silence
    have sigma5 = 0 and get label 0."""
    w = rm.glorot_ffn(0)
    for k in w:
        w[k] = np.full_like(w[k], 1e-6) if k.startswith("W") else np.zeros_like(w[k])
    w["b4"] = np.array([0.0, 1.0, 0.0], np.float32)
    return w


@pytest.fixture(scope="module")
def h():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vad_b200 import runtime
    hd = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    yield hd
    hd.close()


@pytest.fixture(scope="module")
def gh():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vad_b200 import runtime
    hd = runtime.Handle(0, ffn_weights=gated_weights())
    yield hd
    hd.close()


class GatedNoise(object):
    """Per stream, Markov blocks (mean 12 chunks) of digital silence and noise, one chunk per tick."""

    def __init__(self, n, seed):
        self.rng = np.random.default_rng(seed)
        self.on = self.rng.integers(0, 2, n).astype(bool)
        self.n = n

    def chunk(self):
        flip = self.rng.random(self.n) < 1.0 / 12
        self.on ^= flip
        x = self.rng.integers(-3000, 3001, (self.n, 160)).astype(np.int16)
        x[~self.on] = 0
        return x


def check_utterance(S, G, P, labs, rows, bounds, tail):
    """One utterance of one stream: per-tick labels / rows / bounds and its end tail, against the oracle."""
    D = delay(S, G, P)
    lab = labs[labs != 255]
    got = rows[rows != 255]
    assert len(got) == max(0, len(lab) - D)
    n_rows = np.cumsum(labs != 255)
    assert np.array_equal(n_rows[rows != 255], np.arange(len(got)) + D + 1)
    assert (bounds[rows == 255] == -1).all()
    tr, tb = tail
    assert len(tr) == min(len(lab), D) and len(tb) == len(tr) + 1
    ref = rs.smooth(lab, S, G, P)
    assert np.array_equal(np.r_[got, tr].astype(np.uint8), ref)
    b = np.r_[bounds[bounds != -1], tb[tb != -1]]
    seg = rs.segments_of(ref)
    assert np.array_equal(b.reshape(-1, 2), seg)
    return lab, seg


def run_ticks(bank, src, T):
    n = bank.n
    labs = np.empty((T, n), np.uint8)
    rows = np.empty((T, n), np.uint8)
    bounds = np.empty((T, n), np.int64)
    for t in range(T):
        labs[t], rows[t], bounds[t] = bank.feed_speech(src.chunk())
    return labs, rows, bounds


# ---- gated noise: every (S, G, P) of the grid against the oracle --------------------------------------------------
@pytest.mark.parametrize("S,G,P", GRID)
def test_gated_noise_equals_oracle(gh, S, G, P):
    from vad_b200.analyser import StreamBank
    n = 300                                   # 10 CTAs of 32 streams, the last partial
    D = delay(S, G, P)
    T = WARM + D + 400
    bank = StreamBank(n, handle=gh)
    assert bank.set_speech(10 * S, 10 * G, 10 * P) == D == bank.bank.speech_delay()
    labs, rows, bounds = run_ticks(bank, GatedNoise(n, S + 7 * G + 31 * P), T)
    tails = bank.end_streams(range(n))
    both = 0
    for s in range(n):
        lab, _ = check_utterance(S, G, P, labs[:, s], rows[:, s], bounds[:, s], tails[s])
        both += bool((lab == 0).any() and (lab == 1).any())
    assert both >= n // 2                     # the pattern holds both labels in most streams
    # the ended streams start a new signal
    lab2, rows2, _ = bank.feed_speech(np.zeros((n, 160), np.int16))
    assert (lab2 == 255).all() and (rows2 == 255).all()


def test_labels_and_logits_unchanged_by_speech(gh, h):
    import torch
    from vad_b200 import runtime
    for hd in (gh, h):
        n, T = 300, 60
        dev = hd.device
        plain = runtime.StreamBankHandle(hd, n)
        sp = runtime.StreamBankHandle(hd, n)
        assert sp.set_speech(25, 10, 3) == 36
        src = GatedNoise(n, 3)
        out = {k: (torch.empty((n,), dtype=torch.uint8, device=dev), torch.empty((n, 3), dtype=torch.float32,
                                                                                    device=dev)) for k in (0, 1)}
        rows = torch.empty((n,), dtype=torch.uint8, device=dev)
        bounds = torch.empty((n,), dtype=torch.int64, device=dev)
        for t in range(T):
            x = torch.from_numpy(src.chunk()).to(dev)
            plain.feed_ptr(x.data_ptr(), out[0][0].data_ptr(), out[0][1].data_ptr())
            if t % 2:
                sp.feed_speech_ptr(x.data_ptr(), out[1][0].data_ptr(), out[1][1].data_ptr(), rows.data_ptr(),
                                   bounds.data_ptr())
            else:
                sp.feed_ptr(x.data_ptr(), out[1][0].data_ptr(), out[1][1].data_ptr())
            torch.cuda.synchronize()
            assert torch.equal(out[0][0], out[1][0])
            assert torch.equal(out[0][1].view(torch.int32), out[1][1].view(torch.int32))
        plain.close()
        sp.close()


# ---- end to end: utterances one after another in each slot --------------------------------------------------------
def utterance_pool():
    cat = list(_signals.catalogue().values())
    syn = [synth_utterance(77, i, n) for i, n in enumerate((16000, 9000, 24000, 3000, 1200, 500, 160 * 9, 20000))]
    pool = [u[:160 * (len(u) // 160)] for u in cat + syn]
    return [u for u in pool if len(u)]


@pytest.mark.parametrize("fe", ["default", "preemph_hamming_thresh"])
@pytest.mark.parametrize("S,G,P", [(25, 10, 3), (0, 0, 0), (5, 3, 30)])
def test_end_to_end_equals_batch_speech_segments(h, fe, S, G, P):
    from vad_b200 import batch
    from vad_b200.analyser import StreamBank
    if fe != "default":
        h.set_frontend(0.97, "hamming")
        h.set_decision_threshold(0.5)
    try:
        pool = utterance_pool()
        n = 6
        queues = [[pool[(s + 3 * k) % len(pool)] for k in range(3)] for s in range(n)]   # 3 utterances a slot
        bank = StreamBank(n, handle=h)
        bank.set_speech(10 * S, 10 * G, 10 * P)
        state = [[0, 0, [], [], []] for _ in range(n)]   # utterance index, chunk index, labels, rows, bounds
        results = {}
        while any(st[0] < 3 for st in state):
            x = np.zeros((n, 160), np.int16)
            for s, st in enumerate(state):
                if st[0] < 3:
                    u = queues[s][st[0]]
                    x[s] = u[160 * st[1]:160 * (st[1] + 1)]
            lab, rows, bounds = bank.feed_speech(x)
            done = []
            for s, st in enumerate(state):
                if st[0] >= 3:
                    continue
                st[2].append(lab[s]); st[3].append(rows[s]); st[4].append(bounds[s])
                st[1] += 1
                if 160 * st[1] == len(queues[s][st[0]]):
                    done.append(s)
            if done:                                          # streams end at different ticks
                for s, tail in zip(done, bank.end_streams(done)):
                    st = state[s]
                    results[(s, st[0])] = (np.array(st[2], np.uint8), np.array(st[3], np.uint8),
                                           np.array(st[4], np.int64), tail)
                    st[0] += 1
                    st[1] = 0
                    st[2], st[3], st[4] = [], [], []
        utts = [queues[s][k] for s in range(n) for k in range(3)]
        ref = batch.speech_segments(utts, handle=h, min_speech_ms=10 * S, min_silence_ms=10 * G, pad_ms=10 * P)
        for i, (s, k) in enumerate([(s, k) for s in range(n) for k in range(3)]):
            labs, rows, bounds, tail = results[(s, k)]
            _, seg = check_utterance(S, G, P, labs, rows, bounds, tail)
            assert np.array_equal(seg, ref[i]), (s, k)
    finally:
        h.set_frontend(0.0, None)
        h.set_decision_threshold(None)


# ---- isolation ---------------------------------------------------------------------------------------------------
def test_ending_half_the_streams_leaves_the_others_untouched(gh):
    from vad_b200.analyser import StreamBank
    n, T = 64, 150
    a, b = StreamBank(n, handle=gh), StreamBank(n, handle=gh)
    a.set_speech(40, 50, 20)
    b.set_speech(40, 50, 20)
    src = GatedNoise(n, 21)
    ended = list(range(0, n, 2))
    for t in range(T):
        x = src.chunk()
        oa, ob = a.feed_speech(x), b.feed_speech(x)
        for u, v in zip(oa, ob):
            assert np.array_equal(u[1::2], v[1::2])
            if t <= 60:
                assert np.array_equal(u, v)
        if t == 60:
            a.end_streams(ended)
        if t == 61:
            assert (oa[0][0::2] == 255).all()


# ---- other behaviour -----------------------------------------------------------------------------------------------
def test_reset_and_set_speech_clear_the_state(gh):
    from vad_b200.analyser import StreamBank
    n = 40
    fresh, used = StreamBank(n, handle=gh), StreamBank(n, handle=gh)
    for how in ("reset", "set_speech"):
        fresh.set_speech(30, 20, 5)
        used.set_speech(30, 20, 5)
        run_ticks(used, GatedNoise(n, 1), 90)
        if how == "reset":
            used.reset()
        else:
            used.set_speech(30, 20, 5)
        got = run_ticks(used, GatedNoise(n, 2), 120)
        ref = run_ticks(fresh, GatedNoise(n, 2), 120)
        for u, v in zip(got, ref):
            assert np.array_equal(u, v), how


def test_graph_zero_copy_and_interleaved_feed_agree(gh):
    from vad_b200.analyser import StreamBank
    n, T = 70, 130
    banks = [StreamBank(n, handle=gh, use_graph=g, zero_copy=z) for g, z in ((True, True), (True, False),
                                                                              (False, True), (False, False))]
    mixed = StreamBank(n, handle=gh)
    for bk in banks + [mixed]:
        assert bk.set_speech(200, 300, 40) == 52       # 20 / 30 / 4 rows
    src = GatedNoise(n, 5)
    for t in range(T):
        x = src.chunk()
        outs = [bk.feed_speech(x) for bk in banks]
        for o in outs[1:]:
            for u, v in zip(o, outs[0]):
                assert np.array_equal(u, v)
        if t % 3 == 1:
            assert np.array_equal(mixed.feed(x), outs[0][0])   # feed() advances the segments too
        else:
            for u, v in zip(mixed.feed_speech(x), outs[0]):
                assert np.array_equal(u, v)
    tails = [bk.end_streams(range(n)) for bk in banks + [mixed]]
    for tl in tails[1:]:
        for (r0, b0), (r1, b1) in zip(tl, tails[0]):
            assert np.array_equal(r0, r1) and np.array_equal(b0, b1)


def test_disable_speech_restores_the_plain_bank(gh):
    from vad_b200.analyser import StreamBank
    n = 33
    a, b = StreamBank(n, handle=gh), StreamBank(n, handle=gh)
    a.set_speech(10, 10, 10)
    run_ticks(a, GatedNoise(n, 8), 30)
    a.disable_speech()
    assert a.bank.speech_delay() == -1 and a.delay == -1
    with pytest.raises(RuntimeError):
        a.feed_speech(np.zeros((n, 160), np.int16))
    src_a, src_b = GatedNoise(n, 9), GatedNoise(n, 9)
    for _ in range(40):
        la, lga = a.feed(src_a.chunk(), want_logits=True)
        lb, lgb = b.feed(src_b.chunk(), want_logits=True)
        assert np.array_equal(la, lb) and np.array_equal(lga.view(np.int32), lgb.view(np.int32))
    assert all(r.size == 0 and bd.size == 0 for r, bd in a.end_streams([0, 5]))   # speech off: a plain reset
    assert (a.feed(np.zeros((n, 160), np.int16))[[0, 5]] == 255).all()


def test_invalid_arguments(gh):
    import torch
    from vad_b200._lib import VadB200Error
    from vad_b200.analyser import StreamBank
    n = 8
    bank = StreamBank(n, handle=gh)
    with pytest.raises(RuntimeError):
        bank.feed_speech(np.zeros((n, 160), np.int16))
    with pytest.raises(ValueError):
        bank.set_speech(min_speech_ms=10010)
    raw = bank.bank
    lib = gh.lib
    for bad in [(1001, 0, 0), (0, 1001, 0), (0, 0, 1001), (-1, 0, 0)]:
        assert lib.vadb200_stream_bank_set_speech(raw._b, 1, *bad, None) == -1
    assert raw.speech_delay() == -1
    x = torch.zeros((n, 160), dtype=torch.int16, device=gh.device)
    lab = torch.empty((n,), dtype=torch.uint8, device=gh.device)
    with pytest.raises(VadB200Error) as e:
        raw.feed_speech_ptr(x.data_ptr(), lab.data_ptr())
    assert e.value.code == -5                    # speech off
    with pytest.raises(VadB200Error) as e:
        raw.end_streams_ptr(0)
    assert e.value.code == -1                    # null mask
    assert raw.set_speech(0, 0, 1000) == 1000
    with pytest.raises(VadB200Error) as e:
        raw.feed_speech_ptr(0, lab.data_ptr())
    assert e.value.code == -1
    with pytest.raises(ValueError):
        bank.end_streams([n])
    torch.cuda.synchronize()
