"""GPU: the resampling ragged bank (vadb200_stream_bank_create_ragged_rate).  Fed source-rate packets of any size,
each stream's rows are bit-identical to the fused fp32 path on the first M(N) samples of vadb200_resample_packed's
output for its whole signal, plus one; 16 kHz is exactly the plain ragged bank; speech bounds, ends, bad lengths,
graph capture and the output buffers behave as on the 16 kHz ragged bank."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_resample import RATES
from test_gpu_segments import GRID
from test_gpu_stream_ragged import bits, catalogue_signals, feed_signals, pack
from test_gpu_stream_speech import GatedNoise, check_utterance, delay, gated_weights
from test_stream_resample_cpu import design, ready

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def h():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vad_b200 import runtime
    from oracle import ref_math as rm
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


def resampled_prefix(h, signals, rate, lengths):
    """vadb200_resample_packed's output for each whole signal (int16 input), cut to M(N) for N = lengths[i]."""
    from vad_b200 import batch
    ys = batch.resample([np.asarray(s, np.int16) for s in signals], rate, handle=h)
    return [np.asarray(y)[:ready(int(n), rate)] for y, n in zip(ys, lengths)]


def offline(h, ys):
    from vad_b200 import batch
    lab, lg = batch.vad_batch([np.r_[y, np.zeros(1, np.int16)] for y in ys], handle=h, want_logits=True)
    return [x.cpu().numpy() for x in lab], [x.cpu().numpy() for x in lg]


def packet_draw(rate, cap, rng):
    up, down, _, K = design(rate)
    sizes = np.array([0, 1, K - 1, K, K + 1, 160 * down // up - 1, 160 * down // up, 160 * down // up + 1, cap])
    return lambda i: int(rng.choice(sizes)) if i % 2 else int(rng.integers(0, cap + 1))


def check_streams(h, bank, signals, rate, got_l, got_g):
    ys = resampled_prefix(h, signals, rate, [len(s) for s in signals])
    ref_l, ref_g = offline(h, ys)
    for i in range(len(signals)):
        assert np.array_equal(got_l[i], ref_l[i]), i
        assert np.array_equal(bits(got_g[i]), bits(ref_g[i])), i


# ---- 1. every rate: the fused fp32 path on the resampled prefix, bit for bit ---------------------------------------
@pytest.mark.parametrize("rate", RATES)
def test_every_rate_equals_the_offline_path(h, rate):
    from vad_b200.analyser import StreamBank
    rng = np.random.default_rng(rate)
    n, cap = 200, rate // 20
    signals = catalogue_signals(n, rate)
    bank = StreamBank(n, handle=h, max_feed_samples=cap, sample_rate=rate)
    up, down, _, _ = design(rate)
    cap16 = -(-cap * up // down)
    assert bank.sample_rate == rate and bank.k == -(-cap16 // 160)
    assert h.lib.vadb200_stream_bank_sample_rate(bank.bank._b) == rate
    got_l, got_g = feed_signals(bank, signals, packet_draw(rate, cap, rng), idle=0.2, rng=rng)
    check_streams(h, bank, signals, rate, got_l, got_g)


# ---- 2. 16 kHz is the plain ragged bank -----------------------------------------------------------------------------
def test_16k_is_the_plain_ragged_bank(h):
    import torch
    from vad_b200 import runtime
    n, cap, dev = 70, 480, h.device
    a, b = runtime.StreamBankHandle(h, n, cap), runtime.StreamBankHandle(h, n, cap, 16000)
    assert h.lib.vadb200_stream_bank_sample_rate(a._b) == h.lib.vadb200_stream_bank_sample_rate(b._b) == 16000
    assert a.max_rows_per_feed() == b.max_rows_per_feed() == 3
    rng = np.random.default_rng(1)
    K = 3
    for t in range(40):
        c = rng.choice([0, 1, 160, 333, 480], size=n)
        flat = torch.from_numpy(rng.integers(-20000, 20000, int(c.sum()) + 1).astype(np.int16)).to(dev)
        off = torch.from_numpy(np.r_[0, np.cumsum(c)].astype(np.int64)).to(dev)
        outs = []
        for bank in (a, b):
            cnt = torch.full((n,), -9, dtype=torch.int32, device=dev)
            lab = torch.full((n, K), 77, dtype=torch.uint8, device=dev)
            lg = torch.full((n, K, 3), -7.0, dtype=torch.float32, device=dev)
            before = h.lib.vadb200_launch_count()
            bank.feed_ragged_ptr(flat.data_ptr(), off.data_ptr(), cnt.data_ptr(), lab.data_ptr(), lg.data_ptr())
            assert h.lib.vadb200_launch_count() == before + 1
            torch.cuda.synchronize()
            outs.append((cnt.cpu().numpy(), lab.cpu().numpy(), bits(lg.cpu().numpy())))
        for x, y in zip(*outs):
            assert np.array_equal(x, y)
    a.close()
    b.close()


# ---- 3. front end and decision threshold ----------------------------------------------------------------------------
def test_front_end_and_threshold_keep_bit_identity(h):
    from vad_b200.analyser import StreamBank
    h.set_frontend(0.97, "hamming")
    h.set_decision_threshold(0.5)
    try:
        rate, n = 44100, 60
        rng = np.random.default_rng(3)
        signals = catalogue_signals(n, 9)
        bank = StreamBank(n, handle=h, max_feed_samples=1764, sample_rate=rate)
        got_l, got_g = feed_signals(bank, signals, packet_draw(rate, 1764, rng), idle=0.2, rng=rng)
        check_streams(h, bank, signals, rate, got_l, got_g)
    finally:
        h.set_frontend(0.0, None)
        h.set_decision_threshold(None)


# ---- 4. speech segments ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate", [8000, 48000])
@pytest.mark.parametrize("S,G,P", [GRID[0], GRID[2], GRID[3], GRID[7]])
def test_speech_bounds_equal_offline_smoothing(gh, rate, S, G, P):
    from vad_b200 import batch
    from vad_b200.analyser import StreamBank
    n = 48
    up, down, _, _ = design(rate)
    D = delay(S, G, P)
    src = GatedNoise(n, S + 7 * G + 31 * P + rate)
    T = (7 + D + 200) * down // up + 2
    sig = np.concatenate([src.chunk() for _ in range(T)], axis=1)
    cap = 3 * 160 * down // up
    bank = StreamBank(n, handle=gh, max_feed_samples=cap, sample_rate=rate)
    assert bank.set_speech(10 * S, 10 * G, 10 * P) == D
    rng = np.random.default_rng(rate + S)
    pos = np.zeros(n, np.int64)
    per = [[[], [], [], []] for _ in range(n)]
    while (pos < sig.shape[1]).any():
        c = rng.choice([0, 1, 160 * down // up, cap, int(rng.integers(0, cap + 1))], size=n)
        x = [sig[i, pos[i]:pos[i] + c[i]] for i in range(n)]
        pos += [len(v) for v in x]
        out = bank.feed_samples_speech(x)
        raw = bank._rows_of(bank.h_bounds.numpy())          # the C level: 16 kHz bounds
        for i in range(n):
            for k, v in enumerate((out[i][0], out[i][1], raw[i], out[i][2])):
                per[i][k].append(v)
    tails = bank.end_streams(range(n))
    raw_tails = bank.d_tail_bounds.cpu().numpy()
    ys = resampled_prefix(gh, list(sig), rate, [sig.shape[1]] * n)
    ref_l, _ = offline(gh, ys)
    for i in range(n):
        labs, rows, b16, bsrc = (np.concatenate(v) for v in per[i])
        assert np.array_equal(labs, ref_l[i]), i
        k = len(tails[i][0])
        _, seg = check_utterance(S, G, P, labs, rows, b16, (tails[i][0], raw_tails[i][:k + 1]))
        want = batch.source_bounds(seg, sig.shape[1], rate).reshape(-1)
        got = np.r_[bsrc[bsrc != -1], tails[i][1][tails[i][1] != -1]]
        assert np.array_equal(got, want), i


# ---- 5. ending streams ----------------------------------------------------------------------------------------------
def test_ending_half_the_streams_leaves_the_others_untouched(h):
    from vad_b200.analyser import StreamBank
    rate, n, cap, T, t_end = 48000, 64, 1440, 50, 20
    rng = np.random.default_rng(5)
    sig = rng.integers(-12000, 12000, (n, cap * T)).astype(np.int16)
    a, b = (StreamBank(n, handle=h, max_feed_samples=cap, sample_rate=rate) for _ in range(2))
    pos = np.zeros(n, np.int64)
    restart = np.zeros(n, np.int64)
    labs = [[] for _ in range(n)]
    for t in range(T):
        c = rng.choice([0, 1, 100, 480, 960, cap], size=n)
        x = [sig[i, pos[i]:pos[i] + c[i]] for i in range(n)]
        pos += c
        oa, ob = a.feed_samples(x), b.feed_samples(x)
        for i in range(n):
            if i % 2 or t <= t_end:
                assert np.array_equal(oa[i], ob[i]), (t, i)
            if t > t_end:
                labs[i].append(oa[i])
        if t == t_end:
            a.end_streams(range(0, n, 2))
            restart[::2] = pos[::2]
    # the ended streams' rows since the end are an offline run of their new signal from scratch
    ended = list(range(0, n, 2))
    ys = resampled_prefix(h, [sig[i, restart[i]:pos[i]] for i in ended], rate, [pos[i] - restart[i] for i in ended])
    ref_l, _ = offline(h, ys)
    for j, i in enumerate(ended):
        assert np.array_equal(np.concatenate(labs[i]), ref_l[j]), i


# ---- 6. bad lengths -------------------------------------------------------------------------------------------------
def test_bad_lengths_leave_the_stream_untouched(h):
    import torch
    from vad_b200 import runtime
    rate, n, cap, T, bad_t = 8000, 40, 400, 30, 9
    dev = h.device
    banks = [runtime.StreamBankHandle(h, n, cap, rate) for _ in range(2)]
    K = banks[0].max_rows_per_feed()
    assert K == 5
    rng = np.random.default_rng(6)
    src = rng.integers(-15000, 15000, (n, T * cap)).astype(np.int16)
    pos = np.zeros(n, np.int64)
    bad = {0: -1, 5: cap + 1, 31: cap + 1, 32: -1}
    for t in range(T):
        c = rng.integers(0, cap + 1, n)
        if t == bad_t:
            c[list(bad)] = 0
        packets = [src[i, pos[i]:pos[i] + c[i]] for i in range(n)]
        pos += c
        outs = []
        for b, bank in enumerate(banks):
            flat, off = pack(packets, bad if (t == bad_t and b == 0) else None)
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
        assert np.array_equal(outs[0][0][good], outs[1][0][good])
        assert np.array_equal(outs[0][1][good], outs[1][1][good])
        assert np.array_equal(bits(outs[0][2][good]), bits(outs[1][2][good]))
    for bank in banks:
        bank.close()


# ---- 7. one graph, launches -----------------------------------------------------------------------------------------
def test_one_graph_serves_every_packet_mix_and_launches_are_counted(h):
    import torch
    from vad_b200.analyser import StreamBank
    rate, n, cap = 48000, 90, 1920
    banks = [StreamBank(n, handle=h, max_feed_samples=cap, sample_rate=rate, use_graph=g, zero_copy=z)
             for g, z in ((True, True), (False, True), (False, False))]
    rng = np.random.default_rng(7)
    sig = rng.integers(-9000, 9000, (n, cap * 40)).astype(np.int16)
    pos = np.zeros(n, np.int64)
    for t in range(40):
        c = rng.choice([0, 480, 960, cap, 1, 333], size=n) if t % 5 else np.full(n, cap)
        x = [sig[i, pos[i]:pos[i] + c[i]] for i in range(n)]
        pos += c
        before = h.lib.vadb200_launch_count()
        outs = [bk.feed_samples(x, want_logits=True) for bk in banks]
        if t > 0:   # the graph was captured on the first tick: replays issue no library launch
            assert h.lib.vadb200_launch_count() - before == 2 * 3
        for o in outs[1:]:
            for i in range(n):
                assert np.array_equal(o[0][i], outs[0][0][i]) and np.array_equal(bits(o[1][i]), bits(outs[0][1][i]))
    assert list(banks[0]._graphs) == [(True, False)]
    before = h.lib.vadb200_launch_count()
    banks[1].end_streams([0, 3])
    assert h.lib.vadb200_launch_count() - before == 2
    torch.cuda.synchronize()


# ---- 8. guard bands -------------------------------------------------------------------------------------------------
def test_outputs_stay_inside_their_buffers(gh):
    import torch
    from vad_b200 import runtime
    rate, n, cap, G = 22050, 45, 2205, 512
    dev = gh.device
    bank = runtime.StreamBankHandle(gh, n, cap, rate)
    K = bank.max_rows_per_feed()
    assert K == -(-(-(-cap * 320 // 441)) // 160)
    bank.set_speech(3, 2, 1)

    def guarded(count, dtype, fill):
        buf = torch.full((count + 2 * G,), fill, dtype=dtype, device=dev)
        return buf, buf[G:G + count]

    rng = np.random.default_rng(8)
    for t in range(25):
        c = rng.integers(0, cap + 1, n)
        c[:3] = cap
        flat = torch.from_numpy(rng.integers(-3000, 3000, int(c.sum()) + 1).astype(np.int16)).to(dev)
        off = torch.from_numpy(np.r_[0, np.cumsum(c)].astype(np.int64)).to(dev)
        bufs = [guarded(n, torch.int32, -9), guarded(n * K, torch.uint8, 77), guarded(n * K * 3, torch.float32, -7.0),
                guarded(n * K, torch.uint8, 77), guarded(n * K, torch.int64, -9)]
        before = gh.lib.vadb200_launch_count()
        bank.feed_ragged_ptr(flat.data_ptr(), off.data_ptr(), *[v.data_ptr() for _, v in bufs])
        assert gh.lib.vadb200_launch_count() == before + 3
        torch.cuda.synchronize()
        for (buf, view), fill in zip(bufs, (-9, 77, -7.0, 77, -9)):
            m = view.numel()
            assert bool((buf[:G] == fill).all()) and bool((buf[G + m:] == fill).all())
        cnt = bufs[0][1].cpu().numpy()
        lab = bufs[1][1].cpu().numpy().reshape(n, K)
        assert ((cnt >= 0) & (cnt <= K)).all()
        for i in range(n):
            assert (lab[i, :cnt[i]] <= 1).all() and (lab[i, cnt[i]:] == 255).all()
    bank.close()


# ---- 9. argument checks ---------------------------------------------------------------------------------------------
def test_argument_checks(gh):
    import torch
    from vad_b200 import runtime
    from vad_b200._lib import VadB200Error
    lib = gh.lib
    for rate in (3999, 16001, 384001, 7):
        out = C.c_void_p(5)
        assert lib.vadb200_stream_bank_create_ragged_rate(gh._h, 4, 100, rate, C.byref(out)) == -2 and not out.value
    for cap in (0, -1, 8001):
        out = C.c_void_p(5)
        assert lib.vadb200_stream_bank_create_ragged_rate(gh._h, 4, cap, 8000, C.byref(out)) == -1 and not out.value
    out = C.c_void_p(5)
    assert lib.vadb200_stream_bank_create_ragged_rate(gh._h, 0, 80, 8000, C.byref(out)) == -1 and not out.value
    bank = runtime.StreamBankHandle(gh, 4, 8000, 8000)           # a whole second at 8 kHz
    assert bank.max_rows_per_feed() == 100
    x = torch.zeros((4, 160), dtype=torch.int16, device=gh.device)
    lab = torch.empty((4,), dtype=torch.uint8, device=gh.device)
    with pytest.raises(VadB200Error) as e:
        bank.feed_ptr(x.data_ptr(), lab.data_ptr())
    assert e.value.code == -5
    torch.cuda.synchronize()
    bank.close()
    with pytest.raises(ValueError):
        runtime.StreamBankHandle(gh, 4, None, 8000)


# ---- 10. full size --------------------------------------------------------------------------------------------------
def test_4096_streams_48k_jitter_mix_against_offline_labels(h):
    from vad_b200 import batch
    from vad_b200.analyser import StreamBank
    from vad_b200.synth import synth_utterance
    rate, n, T = 48000, 4096, 40
    rng = np.random.default_rng(10)
    sig = np.stack([synth_utterance(10, s, 960 * T) for s in range(n)])
    bank = StreamBank(n, handle=h, max_feed_samples=960, sample_rate=rate)
    pos = np.zeros(n, np.int64)
    labs = [[] for _ in range(n)]
    for t in range(T):
        c = rng.choice([0, 480, 960], size=n)
        out = bank.feed_samples([sig[i, pos[i]:pos[i] + c[i]] for i in range(n)])
        pos += c
        for i in range(n):
            labs[i].append(out[i])
    assert bank._graphs
    ys = resampled_prefix(h, list(sig), rate, pos)
    ref = batch.vad_batch([np.r_[y, np.zeros(1, np.int16)] for y in ys], handle=h)
    for i in range(n):
        assert np.array_equal(np.concatenate(labs[i]), ref[i].cpu().numpy()), i
