"""GPU: speech segments and speech audio (vad_segments.cuh) through the C ABI, Plan and vad_b200.batch -- bit for bit
against the run oracle of oracle/ref_segments.py."""
import ctypes as C

import numpy as np
import pytest

from oracle import ref_frontend as rf, ref_math as rm, ref_segments as rs
from vad_b200.synth import synth_utterance

import _signals
from test_segments_cpu import markov_labels

pytestmark = pytest.mark.gpu

GRID = [(0, 0, 0), (1, 1, 1), (25, 10, 3), (2, 1000, 0), (1000, 0, 0), (0, 0, 1000), (1000, 1000, 1000),
        (5, 3, 30)]


def length_for_rows(R):
    """Samples of an utterance with exactly R label rows (T = R + 5 frames)."""
    return 160 * (R + 4) + 401


@pytest.fixture(scope="module")
def h():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vad_b200 import runtime
    hd = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    yield hd
    hd.close()


def label_plan(h, rows, mode=None):
    """A plan with utterances of the given row counts (no PCM is needed for segments)."""
    from vad_b200 import batch, runtime
    lens = [0 if R < 0 else length_for_rows(R) for R in rows]
    offsets = np.zeros(len(lens), np.int64)
    if len(lens) > 1:
        offsets[1:] = np.cumsum([(n + 7) // 8 * 8 for n in lens[:-1]])
    plan = runtime.Plan(h, offsets, np.array(lens, np.int64), runtime.MODE_VAD if mode is None else mode)
    assert list(np.diff(plan.row_offsets)) == [max(R, 0) for R in rows]
    return plan


def check_plan(plan, labels_np, S, G, P):
    import torch
    lab = torch.from_numpy(labels_np).cuda()
    segs, so, sp, sm = plan.speech_segments(lab, 10 * S, 10 * G, 10 * P, want_smoothed=True)
    ro = plan.row_offsets
    ref_sm, ref_g, ref_so, ref_sp = rs.batch([labels_np[ro[u]:ro[u + 1]] for u in range(plan.n_utt)], S, G, P)
    assert np.array_equal(sm.cpu().numpy(), ref_sm)
    assert np.array_equal(so, ref_so) and np.array_equal(sp, ref_sp)
    assert np.array_equal(segs.cpu().numpy(), ref_g)
    return segs, so, sp


@pytest.mark.parametrize("S,G,P", GRID)
def test_random_labels_ragged_plan(h, S, G, P):
    rng = np.random.default_rng(S * 1000003 + G * 1009 + P)
    rows = [0, 1, 2047, 2048, 2049, -1, 5, 4097, 995, 30000, 1, 0]
    plan = label_plan(h, rows)
    mean = [2, 8, 50, 300]
    labels = np.concatenate([markov_labels(rng, max(R, 0), mean[i % 4]) for i, R in enumerate(rows)]).astype(np.uint8)
    check_plan(plan, labels, S, G, P)


@pytest.mark.parametrize("S,G,P", [(25, 10, 3), (1000, 1000, 1000), (0, 0, 0)])
def test_six_hour_utterance(h, S, G, P):
    rng = np.random.default_rng(7)
    rows = [3, 2_200_000, 17]
    plan = label_plan(h, rows)
    labels = np.concatenate([markov_labels(rng, R, 50) for R in rows]).astype(np.uint8)
    check_plan(plan, labels, S, G, P)


def test_alternating_rows_fill_the_segment_bound(h):
    rows = [1, 2, 2049, 10000]
    plan = label_plan(h, rows)
    labels = np.concatenate([(np.arange(R) % 2 == 0).astype(np.uint8) for R in rows])
    segs, so, _ = check_plan(plan, labels, 0, 0, 0)
    assert segs.shape[0] == int(h.lib.vadb200_plan_max_speech_segments(plan._p)) == sum((R + 1) // 2 for R in rows)


def test_labels_never_bridge_utterances(h):
    rows = [100, 100, 100]
    plan = label_plan(h, rows)
    labels = np.zeros(300, np.uint8)
    labels[:98] = 1            # speech up to 2 rows before the edge, silence, speech 2 rows after it
    labels[102:200] = 1
    labels[200:300] = 1        # speech right across the next edge: two segments, not one
    for S, G, P in [(0, 50, 0), (0, 0, 40), (150, 0, 0), (0, 0, 0)]:
        segs, so, _ = check_plan(plan, labels, S, G, P)
        if (S, G, P) != (150, 0, 0):
            assert list(so) == [0, 1, 2, 3]


def test_dataset_plan_and_zero_rows(h):
    from vad_b200 import runtime
    import torch
    rng = np.random.default_rng(3)
    plan = label_plan(h, [10, 2500, 0], mode=runtime.MODE_DATASET)
    check_plan(plan, markov_labels(rng, 2510, 20), 3, 3, 3)
    empty = label_plan(h, [0, -1, 0])                        # 0 rows: offsets still written, all zero
    segs, so, sp, sm = empty.speech_segments(torch.zeros(0, dtype=torch.uint8, device="cuda"), 100, 100, 100,
                                             want_smoothed=True)
    assert segs.shape == (0, 2) and list(so) == [0, 0, 0, 0] and list(sp) == [0, 0, 0, 0]
    none = label_plan(h, [])
    _, so, sp, _ = none.speech_segments(torch.zeros(0, dtype=torch.uint8, device="cuda"))
    assert list(so) == [0] and list(sp) == [0]


def test_all_params_zero_give_raw_runs(h):
    import torch
    rng = np.random.default_rng(11)
    rows = [700, 3000, 1]
    plan = label_plan(h, rows)
    labels = markov_labels(rng, sum(rows), 6)
    segs, so, sp, sm = plan.speech_segments(torch.from_numpy(labels).cuda(), want_smoothed=True)
    assert np.array_equal(sm.cpu().numpy(), (labels != 0).astype(np.uint8))
    ro = plan.row_offsets
    raw = [rs.segments_of((labels[ro[u]:ro[u + 1]] != 0).astype(np.uint8)) for u in range(3)]
    assert np.array_equal(segs.cpu().numpy(), np.concatenate(raw))


# ---- end to end: fused VAD labels -> segments -> speech audio ------------------------------------------------
def run_e2e(h, utts, S, G, P, theta=None, preemph=0.0, window=None):
    import torch
    from vad_b200 import batch, runtime
    flat, off, ln = batch.pack_utterances(utts)
    plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
    pcm = flat.cuda()
    labels, _, _ = plan.vad(pcm)
    segs, so, sp, sm = plan.speech_segments(labels, 10 * S, 10 * G, 10 * P, want_smoothed=True)
    audio = plan.gather_speech(pcm, segs, so, sp).cpu().numpy()
    lab = labels.cpu().numpy()
    ro = plan.row_offsets
    segs = segs.cpu().numpy()
    for u, x in enumerate(utts):
        dl = lab[ro[u]:ro[u + 1]]
        ref_s, ref_g = rs.speech_segments(dl, S, G, P)
        g = segs[so[u]:so[u + 1]]
        assert np.array_equal(g, ref_g)
        assert np.array_equal(audio[sp[u]:sp[u + 1]], rs.speech_audio(x, ref_g))
        assert np.array_equal(audio[sp[u]:sp[u + 1]], flat.numpy()[np.r_[tuple(slice(off[u] + s, off[u] + e)
                                                                                for s, e in g)] if len(g) else []])
        _, _, _, ol = rf.vad_utterance(x, rm.glorot_ffn(0), preemph=preemph, window=window, threshold=theta)
        if np.array_equal(ol, dl):
            assert np.array_equal(rs.speech_segments(ol, S, G, P)[1], g)
    return audio


@pytest.mark.parametrize("impl", ["tc16", "tc", "fp32"])
@pytest.mark.parametrize("S,G,P", [(0, 0, 0), (25, 10, 3), (3, 30, 8)])
def test_end_to_end_catalogue_and_synthetic(h, impl, S, G, P):
    h.set_ffn_impl(impl)
    try:
        utts = list(_signals.catalogue().values())
        utts += [synth_utterance(91, i, n) for i, n in enumerate((401, 1041, 16000 * 3 + 5, 7777, 160000))]
        run_e2e(h, utts, S, G, P)
    finally:
        h.set_ffn_impl("tc16")


def test_end_to_end_front_end_and_threshold(h):
    h.set_frontend(0.97, "hamming")
    h.set_decision_threshold(0.5)
    try:
        utts = list(_signals.catalogue().values())[:8] + [synth_utterance(5, i, 20000 + 999 * i) for i in range(4)]
        run_e2e(h, utts, 25, 10, 3, theta=0.5, preemph=0.97, window=np.hamming(400))
    finally:
        h.set_frontend(0.0, None)
        h.set_decision_threshold(None)


def test_batch_api(h):
    from vad_b200 import batch
    utts = [synth_utterance(44, i, n) for i, n in enumerate((16000, 32000 + 11, 401, 0, 48000))]
    segs = batch.speech_segments(utts, handle=h, min_speech_ms=250, min_silence_ms=100, pad_ms=30)
    audio = batch.extract_speech(utts, handle=h, min_speech_ms=250, min_silence_ms=100, pad_ms=30)
    labels = batch.vad_batch(utts, handle=h)
    assert len(segs) == len(audio) == len(utts)
    for x, g, a, la in zip(utts, segs, audio, labels):
        _, ref = rs.speech_segments(la.cpu().numpy(), 25, 10, 3)
        assert np.array_equal(g, ref)
        assert a.dtype == np.int16 and np.array_equal(a, rs.speech_audio(x, ref))
    with pytest.raises(ValueError):
        batch.speech_segments(utts, handle=h, pad_ms=10001)


# ---- behaviour ------------------------------------------------------------------------------------------------
def raw_call(h, plan, labels, S, G, P, segs, so, sp, ws, ws_bytes=None, stream=None, smoothed=None):
    from vad_b200.runtime import _ptr
    return h.lib.vadb200_plan_speech_segments(plan._p, _ptr(labels), S, G, P, _ptr(smoothed), _ptr(segs), _ptr(so),
                                              _ptr(sp), _ptr(ws), ws.numel() if ws_bytes is None else ws_bytes,
                                              stream if stream is not None else h.stream)


def test_guard_bands_and_capacity(h):
    import torch
    from vad_b200 import batch, runtime
    from vad_b200.runtime import _ptr
    utts = [synth_utterance(8, i, n) for i, n in enumerate((16000, 30011, 5000))]
    flat, off, ln = batch.pack_utterances(utts)
    plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
    pcm = flat.cuda()
    labels, _, _ = plan.vad(pcm)
    labels.copy_(torch.from_numpy(markov_labels(np.random.default_rng(2), plan.total_rows, 9)).cuda())
    mx = int(h.lib.vadb200_plan_max_speech_segments(plan._p))
    G = 64                                          # guard elements either side of every output
    segs = torch.full((mx * 2 + 2 * G,), -777, dtype=torch.int64, device="cuda")
    offs = torch.full((2 * (plan.n_utt + 1) + 4 * G,), -777, dtype=torch.int64, device="cuda")
    sm = torch.full((plan.total_rows + 2 * G,), 99, dtype=torch.uint8, device="cuda")
    ws = torch.empty(int(h.lib.vadb200_plan_speech_workspace_bytes(plan._p)), dtype=torch.uint8, device="cuda")
    so_v, sp_v = offs[G:G + plan.n_utt + 1], offs[3 * G + plan.n_utt + 1:3 * G + 2 * plan.n_utt + 2]
    assert raw_call(h, plan, labels, 5, 3, 2, segs[G:], so_v, sp_v, ws, smoothed=sm[G:]) == 0
    so, sp = so_v.cpu().numpy(), sp_v.cpu().numpy()
    k = int(so[-1])
    s_np = segs.cpu().numpy()
    assert np.all(s_np[:G] == -777) and np.all(s_np[G + 2 * k:] == -777)
    o_np = offs.cpu().numpy()
    assert np.all(o_np[:G] == -777) and np.all(o_np[G + plan.n_utt + 1:3 * G + plan.n_utt + 1] == -777)
    assert np.all(o_np[3 * G + 2 * plan.n_utt + 2:] == -777)
    sm_np = sm.cpu().numpy()
    assert np.all(sm_np[:G] == 99) and np.all(sm_np[G + plan.total_rows:] == 99)
    seg_t = segs[G:G + 2 * k].view(k, 2)
    full = plan.gather_speech(pcm, seg_t, so, sp).cpu().numpy()
    total = int(sp[-1])
    assert total > 1000
    for cap in (total, total - 1, total - 8, total - 161, 3, 0):
        out = torch.full((total + 2 * 64,), -31111, dtype=torch.int16, device="cuda")
        body = out[64:]                                  # 128-byte offset: still 16-byte aligned
        assert h.lib.vadb200_plan_gather_speech(plan._p, _ptr(pcm), pcm.numel(), _ptr(seg_t), _ptr(so_v), _ptr(sp_v),
                                                _ptr(body), cap, h.stream) == 0
        o = out.cpu().numpy()
        assert np.all(o[:64] == -31111) and np.all(o[64 + cap:] == -31111)
        assert np.array_equal(o[64:64 + cap], full[:cap])


def test_two_streams_and_graph_replay(h):
    import torch
    from vad_b200 import runtime
    rng = np.random.default_rng(5)
    rows = [995] * 50 + [5000, 1]
    planA, planB = label_plan(h, rows), label_plan(h, rows)
    labels = torch.from_numpy(markov_labels(rng, sum(rows), 50)).cuda()
    ref = check_plan(planA, labels.cpu().numpy(), 25, 10, 3)
    outs = []
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    bufs = []
    for plan in (planA, planB):
        mx = int(h.lib.vadb200_plan_max_speech_segments(plan._p))
        ws = torch.empty(int(h.lib.vadb200_plan_speech_workspace_bytes(plan._p)), dtype=torch.uint8, device="cuda")
        bufs.append((torch.empty((mx, 2), dtype=torch.int64, device="cuda"),
                     torch.empty(plan.n_utt + 1, dtype=torch.int64, device="cuda"),
                     torch.empty(plan.n_utt + 1, dtype=torch.int64, device="cuda"), ws))
    torch.cuda.synchronize()
    for _ in range(3):
        for plan, s, (sg, so, sp, ws) in zip((planA, planB), streams, bufs):
            with torch.cuda.stream(s):
                assert raw_call(h, plan, labels, 25, 10, 3, sg, so, sp, ws, stream=C.c_void_p(s.cuda_stream)) == 0
    torch.cuda.synchronize()
    k = int(ref[1][-1])
    for sg, so, sp, _ in bufs:
        assert np.array_equal(sg[:k].cpu().numpy(), ref[0].cpu().numpy())
        assert np.array_equal(so.cpu().numpy(), ref[1]) and np.array_equal(sp.cpu().numpy(), ref[2])
    # CUDA graph: capture segments + gather once, replay, same bytes
    from vad_b200.runtime import _ptr
    plan = planA
    sg, so, sp, ws = bufs[0]
    pcm = torch.from_numpy(synth_utterance(3, 0, int(plan.offsets[-1] + plan.lengths[-1]) + 8)).cuda()
    total = int(ref[2][-1])
    out = torch.empty(total + 8, dtype=torch.int16, device="cuda")
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            cs = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            assert raw_call(h, plan, labels, 25, 10, 3, sg, so, sp, ws, stream=cs) == 0
            assert h.lib.vadb200_plan_gather_speech(plan._p, _ptr(pcm), pcm.numel(), _ptr(sg), _ptr(so), _ptr(sp),
                                                    _ptr(out), out.numel(), cs) == 0
    sg.fill_(-1)
    out.fill_(0)
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(sg[:k].cpu().numpy(), ref[0].cpu().numpy())
    direct = plan.gather_speech(pcm, ref[0], ref[1], ref[2]).cpu().numpy()
    assert np.array_equal(out[:total].cpu().numpy(), direct)
    ro = plan.row_offsets
    p_np = pcm.cpu().numpy()
    segs_np = ref[0].cpu().numpy()
    for u in (0, 49, 50):
        uo = int(plan.offsets[u])
        ga = [p_np[uo + a:uo + b] for a, b in segs_np[ref[1][u]:ref[1][u + 1]]]
        want = np.concatenate(ga) if ga else np.zeros(0, np.int16)
        assert np.array_equal(direct[ref[2][u]:ref[2][u + 1]], want)
    g.reset()


def test_invalid_arguments(h):
    import torch
    from vad_b200 import runtime
    from vad_b200.runtime import _ptr
    E = -1
    plan = label_plan(h, [100, 200])
    labels = torch.zeros(300, dtype=torch.uint8, device="cuda")
    mx = int(h.lib.vadb200_plan_max_speech_segments(plan._p))
    assert mx == 150
    segs = torch.empty((mx + 1, 2), dtype=torch.int64, device="cuda")
    so = torch.empty(3, dtype=torch.int64, device="cuda")
    sp = torch.empty(3, dtype=torch.int64, device="cuda")
    nb = int(h.lib.vadb200_plan_speech_workspace_bytes(plan._p))
    ws = torch.empty(nb + 64, dtype=torch.uint8, device="cuda")
    assert raw_call(h, plan, labels, 0, 0, 0, segs, so, sp, ws) == 0
    for S, G, P in [(-1, 0, 0), (0, 1001, 0), (0, 0, 1001)]:
        assert raw_call(h, plan, labels, S, G, P, segs, so, sp, ws) == E
    assert raw_call(h, plan, labels, 0, 0, 0, segs, so, sp, ws, ws_bytes=nb - 1) == E
    assert raw_call(h, plan, labels, 0, 0, 0, segs, so, sp, ws[1:], ws_bytes=nb) == E      # misaligned workspace
    assert raw_call(h, plan, None, 0, 0, 0, segs, so, sp, ws) == E
    assert raw_call(h, plan, labels, 0, 0, 0, None, so, sp, ws) == E
    assert raw_call(h, plan, labels, 0, 0, 0, segs, None, sp, ws) == E
    assert raw_call(h, plan, labels, 0, 0, 0, segs, so, None, ws) == 0                     # speech offsets nullable
    assert h.lib.vadb200_plan_speech_segments(plan._p, _ptr(labels), 0, 0, 0, None, C.c_void_p(segs.data_ptr() + 4),
                                              _ptr(so), _ptr(sp), _ptr(ws), nb, h.stream) == E
    mf = runtime.Plan(h, plan.offsets, plan.lengths, runtime.MODE_MFCC)
    assert h.lib.vadb200_plan_max_speech_segments(mf._p) == -1
    assert h.lib.vadb200_plan_speech_workspace_bytes(mf._p) == -1
    assert raw_call(h, mf, labels, 0, 0, 0, segs, so, sp, ws) == E
    pcm = torch.zeros(int(plan.offsets[-1] + plan.lengths[-1]) + 16, dtype=torch.int16, device="cuda")
    out = torch.empty(1024, dtype=torch.int16, device="cuda")
    gat = h.lib.vadb200_plan_gather_speech
    assert gat(plan._p, _ptr(pcm), pcm.numel(), _ptr(segs), _ptr(so), _ptr(sp), _ptr(out), 1024, h.stream) == 0
    assert gat(plan._p, _ptr(pcm), pcm.numel(), _ptr(segs), _ptr(so), _ptr(sp), _ptr(out[1:]), 1000, h.stream) == E
    assert gat(plan._p, _ptr(pcm[1:]), pcm.numel() - 1, _ptr(segs), _ptr(so), _ptr(sp), _ptr(out), 1000, h.stream) == E
    assert gat(plan._p, _ptr(pcm), 100, _ptr(segs), _ptr(so), _ptr(sp), _ptr(out), 1000, h.stream) == E
    assert gat(plan._p, _ptr(pcm), pcm.numel(), _ptr(segs), _ptr(so), None, _ptr(out), 1000, h.stream) == E
    assert gat(plan._p, _ptr(pcm), pcm.numel(), _ptr(segs), _ptr(so), _ptr(sp), None, 1000, h.stream) == E
    assert gat(plan._p, _ptr(pcm), pcm.numel(), _ptr(segs), _ptr(so), _ptr(sp), _ptr(out), -1, h.stream) == E
    assert gat(mf._p, _ptr(pcm), pcm.numel(), _ptr(segs), _ptr(so), _ptr(sp), _ptr(out), 1000, h.stream) == E
    torch.cuda.synchronize()
    with pytest.raises(TypeError):
        plan.speech_segments(labels[:10])
