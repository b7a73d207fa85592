"""GPU: the ragged stream bank (vadb200_stream_bank_create_ragged / _feed_ragged).  Fed any packet sizes, including
none, each stream's rows are bit-identical to the fixed bank's and to the fused fp32 path's rows of the same signal;
bad packet lengths leave their stream untouched; speech segments, ends, resets and graph capture behave as on the
fixed bank; nothing is written outside the [n][K] outputs."""
import ctypes as C

import numpy as np
import pytest

from oracle import ref_math as rm

import _signals
from test_gpu_segments import GRID
from test_gpu_stream_speech import GatedNoise, check_utterance, delay, gated_weights

pytestmark = pytest.mark.gpu

WARM = 7


@pytest.fixture(scope="module")
def h():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vad_b200 import runtime
    hd = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    hd.set_ffn_impl("fp32")     # the bank's FFN is FP32: the offline comparison is bit for bit
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


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def feed_signals(bank, signals, draw, want_logits=True, idle=0.0, rng=None):
    """Feed every stream its whole signal in packets of draw(i) samples (a fraction `idle` of the ticks feed nothing);
    returns per stream its concatenated labels and logits."""
    n = len(signals)
    pos = [0] * n
    labs = [[] for _ in range(n)]
    lgs = [[] for _ in range(n)]
    while any(p < len(s) for p, s in zip(pos, signals)):
        chunks = []
        for i, s in enumerate(signals):
            k = 0 if (rng is not None and rng.random() < idle) else min(draw(i), len(s) - pos[i])
            chunks.append(s[pos[i]:pos[i] + k])
            pos[i] += k
        out = bank.feed_samples(chunks, want_logits=True)
        for i in range(n):
            assert len(out[0][i]) <= bank.k
            labs[i].append(out[0][i])
            lgs[i].append(out[1][i])
    return [np.concatenate(x) for x in labs], [np.concatenate(x).reshape(-1, 3) for x in lgs]


def offline(h, signals):
    """The fused fp32 path's rows for utterances of N + 1 samples (the rows a stream has after N samples)."""
    from vad_b200 import batch
    utts = [np.r_[s, np.zeros(1, np.int16)] for s in signals]
    lab, lg = batch.vad_batch(utts, handle=h, want_logits=True)
    return [x.cpu().numpy() for x in lab], [x.cpu().numpy() for x in lg]


def fixed_labels(h, signals):
    """The fixed bank fed each signal's whole 160-sample chunks: its non-255 labels and logits per stream."""
    from vad_b200.analyser import StreamBank
    n, T = len(signals), max(len(s) for s in signals) // 160
    bank = StreamBank(n, handle=h)
    labs, lgs = [], []
    for t in range(T):
        x = np.zeros((n, 160), np.int16)
        for i, s in enumerate(signals):
            if 160 * (t + 1) <= len(s):
                x[i] = s[160 * t:160 * (t + 1)]
        la, lg = bank.feed(x, want_logits=True)
        labs.append(la)
        lgs.append(lg)
    labs, lgs = np.stack(labs), np.stack(lgs)
    return [labs[WARM:len(s) // 160, i] for i, s in enumerate(signals)], \
        [lgs[WARM:len(s) // 160, i] for i, s in enumerate(signals)]


def catalogue_signals(n, seed):
    rng = np.random.default_rng(seed)
    cat = list(_signals.catalogue().values())
    return [cat[i % len(cat)][:len(cat[i % len(cat)]) - int(rng.integers(0, 400))] for i in range(n)]


# ---- 1. uniform 160: the fixed bank, bit for bit ------------------------------------------------------------------
@pytest.mark.parametrize("fe", ["default", "preemph_hamming_thresh"])
def test_uniform_160_equals_the_fixed_bank(h, fe):
    from vad_b200.analyser import StreamBank
    if fe != "default":
        h.set_frontend(0.97, "hamming")
        h.set_decision_threshold(0.5)
    try:
        n, T = 300, 40
        fixed, rag = StreamBank(n, handle=h), StreamBank(n, handle=h, max_feed_samples=160)
        assert rag.k == 1 and rag.bank.max_rows_per_feed() == 1 and fixed.bank.max_rows_per_feed() == -1
        for rnd in range(2):
            src = GatedNoise(n, 11 + rnd)
            for t in range(T):
                x = src.chunk()
                x[::3] = np.random.default_rng(t).integers(-20000, 20000, (len(x[::3]), 160))
                la, lg = fixed.feed(x, want_logits=True)
                ra, rg = rag.feed_samples(list(x), want_logits=True)
                assert [len(r) for r in ra] == [0 if t < WARM else 1] * n
                if t >= WARM:
                    assert np.array_equal(np.concatenate(ra), la)
                    assert np.array_equal(bits(np.concatenate(rg)), bits(lg))
            fixed.reset()
            rag.reset()
    finally:
        h.set_frontend(0.0, None)
        h.set_decision_threshold(None)


# ---- 2, 3. random splits and packet shapes: the fused fp32 path, bit for bit ----------------------------------------
def test_random_splits_equal_the_fused_path(h):
    from vad_b200.analyser import StreamBank
    rng = np.random.default_rng(5)
    n, cap = 300, 1024
    signals = catalogue_signals(n, 6)
    bank = StreamBank(n, handle=h, max_feed_samples=cap)
    assert bank.k == 7
    sizes = np.array([0, 1, 79, 80, 81, 159, 160, 161, 399, 400, 401, cap])
    got_l, got_g = feed_signals(bank, signals, lambda i: int(rng.choice(sizes)) if i % 2 else int(rng.integers(0, cap + 1)),
                                idle=0.2, rng=rng)
    ref_l, ref_g = offline(h, signals)
    fix_l, _ = fixed_labels(h, signals)
    for i in range(n):
        assert np.array_equal(got_l[i], ref_l[i]), i
        assert np.array_equal(bits(got_g[i]), bits(ref_g[i])), i
        assert np.array_equal(got_l[i][:len(fix_l[i])], fix_l[i]), i


@pytest.mark.parametrize("packet", [320, 400, 480, 16000])
def test_packet_shapes_equal_the_fused_path(h, packet):
    from vad_b200.analyser import StreamBank
    n = 40
    signals = catalogue_signals(n, packet)
    bank = StreamBank(n, handle=h, max_feed_samples=packet)
    got_l, got_g = feed_signals(bank, signals, lambda i: packet)
    ref_l, ref_g = offline(h, signals)
    for i in range(n):
        assert np.array_equal(got_l[i], ref_l[i]) and np.array_equal(bits(got_g[i]), bits(ref_g[i])), i


# ---- 4. bad packet lengths ------------------------------------------------------------------------------------------
def pack(packets, bad=None):
    """Samples and offsets [n + 1] of the packets; bad = {stream: length} gives those streams that length in the
    offsets instead of their packet (negative, above the cap, or absurd).  A negative length moves every later packet
    back, so the stream before it must be a bad one that owns enough samples; the packets of good streams never
    overlap."""
    bad = bad or {}
    n = len(packets)
    lens = np.array([bad.get(i, len(x)) for i, x in enumerate(packets)], np.int64)
    off = np.r_[0, np.cumsum(lens)]
    off -= min(0, int(off[1:n].min()))
    good = [i for i in range(n) if i not in bad]
    flat = np.zeros(max(int(off[i]) + len(packets[i]) for i in good) + 1, np.int16)
    used = np.zeros(flat.shape, bool)
    for i in good:
        a, b = int(off[i]), int(off[i]) + len(packets[i])
        assert not used[a:b].any()
        used[a:b] = True
        flat[a:b] = packets[i]
    return flat, off


def test_bad_lengths_leave_the_stream_untouched(h):
    import torch
    from vad_b200 import runtime
    n, cap, T, bad_t = 70, 400, 30, 12
    dev = h.device
    banks = [runtime.StreamBankHandle(h, n, cap) for _ in range(2)]
    K = banks[0].max_rows_per_feed()
    rng = np.random.default_rng(8)
    src = rng.integers(-15000, 15000, (n, T * cap)).astype(np.int16)
    pos = np.zeros(n, np.int64)
    # the first stream absurdly negative, an over-cap one, a CTA's last two (over the cap, then negative), the last
    # stream absurdly long
    bad = {0: -(1 << 40), 3: cap + 1, 30: cap + 8, 31: -7, n - 1: 1 << 62}
    for t in range(T):
        c = rng.integers(0, cap + 1, n)
        if t == bad_t:
            c[list(bad)] = 0                  # what the reference bank sees instead
        packets = [src[i, pos[i]:pos[i] + c[i]] for i in range(n)]
        pos += c
        outs = []
        for b, bank in enumerate(banks):
            flat, off = pack(packets, bad if (t == bad_t and b == 0) else None)
            if t == bad_t and b == 0:
                d = np.diff(off)
                assert d[0] < 0 and d[3] == cap + 1 and d[30] > cap and d[31] == -7 and d[n - 1] > cap
            d_flat, d_off = torch.from_numpy(flat).to(dev), torch.from_numpy(off).to(dev)
            cnt = torch.full((n,), -9, dtype=torch.int32, device=dev)
            lab = torch.full((n, K), 77, dtype=torch.uint8, device=dev)
            lg = torch.full((n, K, 3), -7.0, dtype=torch.float32, device=dev)
            bank.feed_ragged_ptr(d_flat.data_ptr(), d_off.data_ptr(), cnt.data_ptr(), lab.data_ptr(), lg.data_ptr())
            torch.cuda.synchronize()
            outs.append((cnt.cpu().numpy(), lab.cpu().numpy(), lg.cpu().numpy()))
        ids = list(bad) if t == bad_t else []
        good = np.setdiff1d(np.arange(n), ids)
        if ids:
            assert (outs[0][0][ids] == -1).all() and (outs[0][1][ids] == 255).all() and (outs[0][2][ids] == -7.0).all()
        for b, o in enumerate(outs):
            for i in (good if b == 0 else range(n)):
                k = o[0][i]
                assert 0 <= k <= K and (o[1][i, k:] == 255).all() and (o[2][i, k:] == -7.0).all()
        assert np.array_equal(outs[0][0][good], outs[1][0][good])
        assert np.array_equal(outs[0][1][good], outs[1][1][good])
        assert np.array_equal(bits(outs[0][2][good]), bits(outs[1][2][good]))
    for bank in banks:
        bank.close()


# ---- 5. speech segments -------------------------------------------------------------------------------------------
class RaggedGatedNoise(object):
    """GatedNoise's signal, one stream's samples cut into packets of 0 .. 480 samples."""

    def __init__(self, n, seed, T):
        src = GatedNoise(n, seed)
        self.sig = np.concatenate([src.chunk() for _ in range(T)], axis=1)
        self.rng = np.random.default_rng(seed + 1)
        self.pos = np.zeros(n, np.int64)

    def packets(self):
        c = self.rng.choice([0, 160, 320, 480, 17, 400], size=len(self.pos))
        out = [self.sig[i, p:p + k] for i, (p, k) in enumerate(zip(self.pos, c))]
        self.pos += [len(x) for x in out]
        return out

    def done(self):
        return (self.pos >= self.sig.shape[1]).all()


@pytest.mark.parametrize("S,G,P", GRID)
def test_speech_segments_equal_oracle_and_fixed_bank(gh, S, G, P):
    from vad_b200.analyser import StreamBank
    n = 64
    D = delay(S, G, P)
    T = WARM + D + 400
    rag = StreamBank(n, handle=gh, max_feed_samples=480)
    fixed = StreamBank(n, handle=gh)
    assert rag.set_speech(10 * S, 10 * G, 10 * P) == D == fixed.set_speech(10 * S, 10 * G, 10 * P)
    src = RaggedGatedNoise(n, S + 7 * G + 31 * P, T)
    per = [[[], [], []] for _ in range(n)]
    while not src.done():
        for i, o in enumerate(rag.feed_samples_speech(src.packets())):
            assert len(o[0]) == len(o[1]) == len(o[2]) <= 3
            for k in range(3):
                per[i][k].append(o[k])
    tails = rag.end_streams(range(n))
    fl, fr, fb = [], [], []
    for t in range(T):
        a, b, c = fixed.feed_speech(src.sig[:, 160 * t:160 * (t + 1)])
        fl.append(a); fr.append(b); fb.append(c)
    ftails = fixed.end_streams(range(n))
    fl, fr, fb = np.stack(fl), np.stack(fr), np.stack(fb)
    for i in range(n):
        labs, rows, bounds = (np.concatenate(x) for x in per[i])
        check_utterance(S, G, P, labs, rows, bounds, tails[i])
        assert np.array_equal(labs, fl[WARM:, i])
        assert np.array_equal(rows[rows != 255], fr[:, i][fr[:, i] != 255])
        assert np.array_equal(bounds[bounds != -1], fb[:, i][fb[:, i] != -1])
        assert np.array_equal(tails[i][0], ftails[i][0]) and np.array_equal(tails[i][1], ftails[i][1])
    out = rag.feed_samples_speech([np.zeros(480, np.int16)] * n)       # the ended streams start a new signal
    assert all(len(o[0]) == 0 for o in out)


# ---- 6. ending streams --------------------------------------------------------------------------------------------
def test_ending_half_the_streams_leaves_the_others_untouched(gh):
    from vad_b200.analyser import StreamBank
    n, T, t_end = 64, 120, 50
    a, b, fresh = (StreamBank(n, handle=gh, max_feed_samples=500) for _ in range(3))
    for bk in (a, b, fresh):
        bk.set_speech(40, 50, 20)
    src = RaggedGatedNoise(n, 4, 2 * T)
    ended = list(range(0, n, 2))
    for t in range(T):
        x = src.packets()
        if t == t_end:
            x = [np.r_[p, np.ones(37, np.int16)][:500] for p in x]    # samples pending that complete no frame
        oa, ob = a.feed_samples_speech(x), b.feed_samples_speech(x)
        for i in range(n):
            if i % 2 or t <= t_end:
                assert all(np.array_equal(u, v) for u, v in zip(oa[i], ob[i])), (t, i)
        if t > t_end:     # the ended streams are new signals: as a fresh bank fed from the end on
            of = fresh.feed_samples_speech([x[i] if i % 2 == 0 else np.zeros(0, np.int16) for i in range(n)])
            for i in ended:
                assert all(np.array_equal(u, v) for u, v in zip(oa[i], of[i])), (t, i)
        if t == t_end:
            a.end_streams(ended)


# ---- 7. graph capture ----------------------------------------------------------------------------------------------
def test_one_graph_serves_every_packet_mix(h):
    from vad_b200.analyser import StreamBank
    n = 90
    banks = [StreamBank(n, handle=h, max_feed_samples=640, use_graph=g, zero_copy=z)
             for g, z in ((True, True), (False, True), (False, False), (True, False))]
    rng = np.random.default_rng(2)
    sig = rng.integers(-9000, 9000, (n, 640 * 60)).astype(np.int16)
    pos = np.zeros(n, np.int64)
    for t in range(60):
        c = rng.choice([0, 160, 320, 640, 1, 333], size=n) if t % 5 else np.full(n, 640)
        x = [sig[i, pos[i]:pos[i] + c[i]] for i in range(n)]
        pos += c
        outs = [bk.feed_samples(x, want_logits=True) for bk in banks]
        for o in outs[1:]:
            for i in range(n):
                assert np.array_equal(o[0][i], outs[0][0][i]) and np.array_equal(bits(o[1][i]), bits(outs[0][1][i]))
    assert list(banks[0]._graphs) == [(True, False)]


# ---- 8, 9, 10. buffers, launches, bank kinds ------------------------------------------------------------------------
def test_outputs_stay_inside_their_buffers_and_one_launch_per_feed(gh):
    import torch
    from vad_b200 import runtime
    n, cap, G = 45, 700, 512
    dev = gh.device
    bank = runtime.StreamBankHandle(gh, n, cap)
    K = bank.max_rows_per_feed()
    assert K == 5
    bank.set_speech(3, 2, 1)

    def guarded(count, dtype, fill):
        buf = torch.full((count + 2 * G,), fill, dtype=dtype, device=dev)
        return buf, buf[G:G + count]

    rng = np.random.default_rng(4)
    for t in range(25):
        c = rng.integers(0, cap + 1, n)
        c[:3] = cap
        flat = torch.from_numpy(rng.integers(-3000, 3000, int(c.sum()) + 1).astype(np.int16)).to(dev)
        off = torch.from_numpy(np.r_[0, np.cumsum(c)].astype(np.int64)).to(dev)
        bufs = [guarded(n, torch.int32, -9), guarded(n * K, torch.uint8, 77), guarded(n * K * 3, torch.float32, -7.0),
                guarded(n * K, torch.uint8, 77), guarded(n * K, torch.int64, -9)]
        before = gh.lib.vadb200_launch_count()
        bank.feed_ragged_ptr(flat.data_ptr(), off.data_ptr(), *[v.data_ptr() for _, v in bufs])
        assert gh.lib.vadb200_launch_count() == before + 1
        torch.cuda.synchronize()
        for (buf, view), fill in zip(bufs, (-9, 77, -7.0, 77, -9)):
            m = view.numel()
            assert bool((buf[:G] == fill).all()) and bool((buf[G + m:] == fill).all())
        cnt = bufs[0][1].cpu().numpy()
        lab, rows, bnd = (bufs[k][1].cpu().numpy().reshape(n, K) for k in (1, 3, 4))
        lg = bufs[2][1].cpu().numpy().reshape(n, K, 3)
        assert ((cnt >= 0) & (cnt <= K)).all()
        for i in range(n):
            k = cnt[i]
            assert (lab[i, :k] <= 1).all() and (lab[i, k:] == 255).all()
            assert (rows[i, k:] == 255).all() and (bnd[i, k:] == -1).all() and (rows[i, :k] != 77).all()
            assert (lg[i, k:] == -7.0).all() and not (lg[i, :k] == -7.0).any()
    bank.close()


def test_wrong_bank_kind_is_a_state_error(gh):
    import torch
    from vad_b200 import runtime
    from vad_b200._lib import VadB200Error
    n = 8
    dev = gh.device
    fixed, rag = runtime.StreamBankHandle(gh, n), runtime.StreamBankHandle(gh, n, 320)
    x = torch.zeros((n + 1, 320), dtype=torch.int16, device=dev)    # room for the feed from x + 1 sample below
    off = torch.arange(n + 1, dtype=torch.int64, device=dev) * 320
    cnt = torch.empty((n,), dtype=torch.int32, device=dev)
    lab = torch.empty((n, 2), dtype=torch.uint8, device=dev)
    rows = torch.empty((n, 2), dtype=torch.uint8, device=dev)
    bnd = torch.empty((n, 2), dtype=torch.int64, device=dev)
    calls = [lambda: rag.feed_ptr(x.data_ptr(), lab.data_ptr()),
             lambda: fixed.feed_ragged_ptr(x.data_ptr(), off.data_ptr(), cnt.data_ptr(), lab.data_ptr()),
             lambda: rag.feed_ragged_ptr(x.data_ptr(), off.data_ptr(), cnt.data_ptr(), lab.data_ptr(), 0,
                                         rows.data_ptr()),                         # speech off
             lambda: rag.feed_ragged_ptr(x.data_ptr(), off.data_ptr(), cnt.data_ptr(), lab.data_ptr(), 0, 0,
                                         bnd.data_ptr())]
    for call in calls:
        with pytest.raises(VadB200Error) as e:
            call()
        assert e.value.code == -5
    rag.set_speech(0, 0, 0)
    fixed.set_speech(0, 0, 0)
    with pytest.raises(VadB200Error) as e:
        rag.feed_speech_ptr(x.data_ptr(), lab.data_ptr())
    assert e.value.code == -5
    with pytest.raises(VadB200Error) as e:
        fixed.feed_ragged_ptr(x.data_ptr(), off.data_ptr(), cnt.data_ptr(), lab.data_ptr(), 0, rows.data_ptr())
    assert e.value.code == -5
    with pytest.raises(VadB200Error) as e:
        rag.feed_ragged_ptr(x.data_ptr() + 1, off.data_ptr(), cnt.data_ptr(), lab.data_ptr())
    assert e.value.code == -1                                                    # odd sample address
    rag.feed_ragged_ptr(x.data_ptr() + 2, off.data_ptr(), cnt.data_ptr(), lab.data_ptr(), 0, rows.data_ptr(),
                        bnd.data_ptr())                                          # 2-byte aligned is enough
    assert rag.max_rows_per_feed() == 2 and fixed.max_rows_per_feed() == -1
    out = C.c_void_p()
    assert gh.lib.vadb200_stream_bank_create_ragged(gh._h, n, 16001, C.byref(out)) == -1 and not out.value
    torch.cuda.synchronize()
    fixed.close()
    rag.close()


# ---- 11. full size ------------------------------------------------------------------------------------------------
def test_4096_streams_jitter_mix_against_offline_labels(h):
    from vad_b200 import batch
    from vad_b200.analyser import StreamBank
    from vad_b200.synth import synth_utterance
    n, T = 4096, 60
    rng = np.random.default_rng(41)
    sig = np.stack([synth_utterance(41, s, 320 * T) for s in range(n)])
    bank = StreamBank(n, handle=h, max_feed_samples=320)
    pos = np.zeros(n, np.int64)
    labs = [[] for _ in range(n)]
    for t in range(T):
        c = rng.choice([0, 160, 320], size=n)
        out = bank.feed_samples([sig[i, pos[i]:pos[i] + c[i]] for i in range(n)])
        pos += c
        for i in range(n):
            labs[i].append(out[i])
    assert bank._graphs
    ref = batch.vad_batch([np.r_[sig[i, :pos[i]], np.zeros(1, np.int16)] for i in range(n)], handle=h)
    for i in range(n):
        got = np.concatenate(labs[i])
        assert len(got) == rm.n_outputs(int(pos[i]) + 1)
        assert np.array_equal(got, ref[i].cpu().numpy()), i
