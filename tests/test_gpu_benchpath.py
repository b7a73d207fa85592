"""GPU parity on the paths the bench and BASELINE.json's configs actually run (through the C ABI):

  cfg3 layout  -- >= 1200 x 10 s utterances, one 997-frame segment per utterance (32 steps, the
                  288-slot MFCC ring wraps three times), as in `python bench.py`
  cfg2         -- MFCC-only at the configured 1024 x 10 s
  cfg5         -- >= 2048 ragged 2-30 s utterances, dataset rows (deltas + delta-deltas) and VAD,
                  segments at the 2048-frame cap
  cfg4         -- 4096 streams in 10 ms chunks against the offline labels
  FEAT_DATASET -- the dataset recipe inside the VAD kernel
  sharding     -- N disjoint shards reproduce the 1-shard labels byte for byte
  threads      -- two host threads x two handles with different classifiers

Sizes the oracle cannot cover in seconds are checked on sampled utterances plus
size-independent properties (duplicates give identical rows, batch position does not matter).
"""
import threading

import numpy as np
import pytest

from oracle import ref_math as rm
from vad_b200.synth import synth_utterance
from _parity import mfcc_close, rows_close, check_vad, decisive_rows, LOGIT_ATOL, LOGIT_RTOL

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hw():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vad_b200 import runtime
    w = rm.glorot_ffn(0)
    h = runtime.Handle(ffn_weights=w)          # private handle: nothing here touches the default one
    yield h, w
    h.close()


def _uniform_batch(h, n_utt, L, seed):
    from vad_b200 import batch
    off, ln, stride = batch.uniform_layout(n_utt, L)
    pcm = h.synth_pcm(n_utt, L, seed=seed, first_utt=0, utt_stride=stride)
    return pcm, off, ln, stride


@pytest.mark.parametrize("impl", ["tc16", "tc", "fp32"])
def test_cfg3_bench_layout_one_segment_per_utterance(hw, impl):
    """The bench's decomposition: every 10 s utterance is ONE 997-frame segment (32 steps, 8 block
    phases, ring wraps).  1200 utterances = 1.19 M rows; 10 sampled utterances against the oracle:
    labels, logits, analyser features, dataset rows and MFCCs."""
    import torch
    from vad_b200 import runtime
    h, w = hw
    h.set_ffn_impl(impl)
    n_utt, L, seed = 1200, 160000, 4242
    pcm, off, ln, stride = _uniform_batch(h, n_utt, L, seed)
    h.set_plan_segment_frames(1024)
    try:
        vplan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
        dplan = runtime.Plan(h, off, ln, runtime.MODE_DATASET)
        mplan = runtime.Plan(h, off, ln, runtime.MODE_MFCC)
    finally:
        h.set_plan_segment_frames(0)
    assert vplan.segment_frames == 1024 and vplan.segment_count == n_utt      # one segment per utterance
    assert vplan.total_rows == n_utt * 993 and mplan.total_rows == n_utt * 998
    labels, logits, feats = vplan.vad(pcm, want_logits=True, want_feats=True)
    labels_only, _, _ = vplan.vad(pcm)                                         # the bench's launch (labels only)
    assert torch.equal(labels, labels_only)
    rows = dplan.mfcc(pcm).view(n_utt, 993, 39)
    mf = mplan.mfcc(pcm).view(n_utt, 998, 13)
    labels = labels.view(n_utt, 993)
    logits = logits.view(n_utt, 993, 3)
    feats = feats.view(n_utt, 993, 39)
    for u in (0, 1, 147, 295, 296, 599, 777, 1023, 1198, 1199):
        host = synth_utterance(seed, u, L)
        c = rm.mfcc_utterance(host)
        assert mfcc_close(mf[u].cpu().numpy(), c)
        assert rows_close(rows[u].cpu().numpy(), rm.dataset_features(c))
        check_vad(labels[u].cpu().numpy(), logits[u].cpu().numpy(), host, w)
        ref_f = rm.analyser_features(c)
        sig = np.lib.stride_tricks.sliding_window_view(c, 5, axis=0)[: c.shape[0] - 5].std(axis=2)
        tol = 3e-4 + 2e-4 / np.maximum(np.tile(sig, 3), 1e-12)                  # z = (c - mu) / sigma5
        assert np.all(np.abs(feats[u].cpu().numpy() - ref_f) <= tol)
    # automatic segmentation (shorter segments) gives byte-identical labels
    aplan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
    assert aplan.segment_frames < 1024 and aplan.segment_count > n_utt
    assert torch.equal(aplan.vad(pcm)[0].view(n_utt, 993), labels)
    h.set_ffn_impl("tc16")


def test_cfg2_mfcc_only_at_1024_utterances(hw):
    import torch
    from vad_b200 import runtime
    h, _ = hw
    n_utt, L, seed = 1024, 160000, 2
    pcm, off, ln, stride = _uniform_batch(h, n_utt, L, seed)
    body = pcm[: n_utt * stride].view(n_utt, stride)
    body[900] = body[17]                                                       # duplicate utterance
    plan = runtime.Plan(h, off, ln, runtime.MODE_MFCC)
    out = plan.mfcc(pcm).view(n_utt, 998, 13)
    assert plan.total_rows == 1021952
    assert torch.equal(out[900], out[17])
    assert bool(torch.isfinite(out).all())
    for u in (0, 17, 511, 512, 1023):
        assert mfcc_close(out[u].cpu().numpy(), rm.mfcc_utterance(synth_utterance(seed, u, L)))
    # end-to-end host pipeline (vadb200_mfcc_host) returns the same rows
    host_pcm = pcm.cpu().pin_memory()
    h.set_host_chunk_samples(40 * 160000)
    try:
        got = plan.mfcc_host(host_pcm)
    finally:
        h.set_host_chunk_samples(32 << 20)
    assert torch.equal(got, out.view(-1, 13).cpu())


def test_cfg5_ragged_2_to_30s_dataset_rows_and_vad(hw):
    """configs[4]: lengths uniform in [2 s, 30 s], seed 7, deltas + delta-deltas, packed.  2048 utterances
    (the oracle covers the longest, shortest and median ones)."""
    import torch
    from vad_b200 import runtime
    h, w = hw
    n_utt, seed = 2048, 7
    rng = np.random.default_rng(seed)
    lens = rng.integers(32000, 480001, size=n_utt).astype(np.int64)
    lens[5], lens[6] = 480000, 32000                                           # both extremes present
    stride = 480000
    off = np.arange(n_utt, dtype=np.int64) * stride
    pcm = h.synth_pcm(n_utt, stride, seed=seed, first_utt=0, utt_stride=stride)
    h.set_plan_segment_frames(2048)       # what >= 8192 utterances get automatically: 20-30 s utterances hit the cap
    try:
        dplan = runtime.Plan(h, off, lens, runtime.MODE_DATASET)
        vplan = runtime.Plan(h, off, lens, runtime.MODE_VAD)
    finally:
        h.set_plan_segment_frames(0)
    assert dplan.segment_frames == 2048 and dplan.segment_count > n_utt
    rows = dplan.mfcc(pcm)
    labels, logits, _ = vplan.vad(pcm, want_logits=True)
    aplan = runtime.Plan(h, off, lens, runtime.MODE_VAD)                       # automatic (shorter) segments
    assert aplan.segment_frames < 2048
    assert torch.equal(aplan.vad(pcm)[0], labels)
    ro = dplan.row_offsets
    assert np.array_equal(np.diff(ro), [rm.n_outputs(int(n)) for n in lens])
    order = np.argsort(lens)
    for u in (5, 6, int(order[n_utt // 2]), int(order[-2]), int(order[1]), 2047):
        host = synth_utterance(seed, u, int(lens[u]))
        c = rm.mfcc_utterance(host)
        assert rows_close(rows[ro[u]:ro[u + 1]].cpu().numpy(), rm.dataset_features(c))
        check_vad(labels[ro[u]:ro[u + 1]].cpu().numpy(), logits[ro[u]:ro[u + 1]].cpu().numpy(), host, w)
    assert bool(torch.isfinite(rows).all())


def test_feat_dataset_inside_vad_kernel_and_windows(hw):
    """VADB200_FEAT_DATASET through vad_packed (both FFN implementations) and vad_windows."""
    from vad_b200 import batch, runtime
    h, w = hw
    utts = [synth_utterance(19, i, n) for i, n in enumerate((16000, 48017, 160000, 2001))]
    flat, off, ln = batch.pack_utterances(utts)
    pcm = flat.to(h.device)
    for impl in ("tc16", "tc", "fp32"):
        h.set_ffn_impl(impl)
        plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
        labels, logits, feats = plan.vad(pcm, want_logits=True, want_feats=True, feat_mode=runtime.FEAT_DATASET)
        ro = plan.row_offsets
        for i, u in enumerate(utts):
            la, lo = labels[ro[i]:ro[i + 1]].cpu().numpy(), logits[ro[i]:ro[i + 1]].cpu().numpy()
            check_vad(la, lo, u, w, mode="dataset")
            ref_rows = rm.dataset_features(rm.mfcc_utterance(u))
            assert rows_close(feats[ro[i]:ro[i + 1]].cpu().numpy(), ref_rows)
    h.set_ffn_impl("tc16")
    c = rm.mfcc_utterance(utts[1])
    win = np.lib.stride_tricks.sliding_window_view(c, 5, axis=0)[: c.shape[0] - 5].transpose(0, 2, 1)
    la, lo, fe = h.vad_windows(np.ascontiguousarray(win, dtype=np.float32), runtime.FEAT_DATASET, want_feats=True)
    ref_f = rm.dataset_features(c)
    ref_lo, _ = rm.ffn_forward(ref_f, w)
    assert rows_close(fe.cpu().numpy(), ref_f)
    assert np.all(np.abs(lo.cpu().numpy() - ref_lo) <= LOGIT_ATOL + LOGIT_RTOL * np.abs(ref_lo))
    dec = decisive_rows(ref_lo)
    assert np.array_equal(la.cpu().numpy()[dec], rm.decide(ref_lo)[dec])


def test_disjoint_shards_reproduce_single_plan_labels(hw):
    """SURVEY 4(iv): sharding must not change results.  Contiguous and LPT-balanced shards of a ragged
    batch, each run as its own plan on its own buffer, give the single-plan labels byte for byte."""
    import torch
    from vad_b200 import batch, runtime, shard
    h, _ = hw
    rng = np.random.default_rng(3)
    lens = rng.integers(300, 90000, size=97)
    utts = [synth_utterance(23, i, int(n)) for i, n in enumerate(lens)]
    flat, off, ln = batch.pack_utterances(utts)
    plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
    base = plan.vad(flat.to(h.device))[0].cpu()
    ro = plan.row_offsets
    for world in (2, 3, 8):
        parts = [np.arange(*shard.shard_contiguous(len(utts), r, world)) for r in range(world)]
        for idx_sets in (parts, shard.shard_balanced(lens, world)):
            for idx in idx_sets:
                sub = [utts[i] for i in idx]
                f2_, o2, l2 = batch.pack_utterances(sub)
                p2 = runtime.Plan(h, o2, l2, runtime.MODE_VAD)
                got = p2.vad(f2_.to(h.device))[0].cpu()
                want = torch.cat([base[ro[i]:ro[i + 1]] for i in idx]) if len(idx) else base[:0]
                assert torch.equal(got, want)


def test_one_plan_on_two_streams_concurrently(hw):
    """ADVICE r1: each launch of a plan takes its own self-resetting work counter, so the same plan can be
    in flight on several streams (and back to back) without skipping segments."""
    import torch
    from vad_b200 import runtime
    h, _ = hw
    n_utt, L = 96, 160000
    pcm, off, ln, _ = _uniform_batch(h, n_utt, L, 31)
    plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
    base = plan.vad(pcm)[0].clone()
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=h.device) for _ in range(4)]
    outs = [torch.full_like(base, 77) for _ in range(12)]
    for i, o in enumerate(outs):
        with torch.cuda.stream(streams[i % 4]):
            plan.vad(pcm, labels=o)
    torch.cuda.synchronize()
    for o in outs:
        assert torch.equal(o, base)
    # 40 back-to-back launches on one stream wrap the counter ring twice
    for _ in range(40):
        plan.vad(pcm, labels=outs[0])
    torch.cuda.synchronize()
    assert torch.equal(outs[0], base)


def test_two_threads_two_handles_different_classifiers(hw):
    """SURVEY 8(b) 'no hidden global state': two host threads drive two handles with different FFN weights
    on the same device, 200 iterations each; every row of every iteration is checked."""
    import torch
    from vad_b200 import batch, runtime
    h, w = hw
    results = {}

    def worker(name, seed, impl):
        try:
            torch.cuda.set_device(h.device)
            ww = rm.glorot_ffn(seed)
            hh = runtime.Handle(h.device.index, ffn_weights=ww)
            hh.set_ffn_impl(impl)
            utts = [synth_utterance(seed, i, 16000 + 777 * i) for i in range(5)]
            flat, off, ln = batch.pack_utterances(utts)
            st = torch.cuda.Stream(device=h.device)
            with torch.cuda.stream(st):
                pcm = flat.to(h.device)
                plan = runtime.Plan(hh, off, ln, runtime.MODE_VAD)
                x = np.random.default_rng(seed).standard_normal((64, 39)).astype(np.float32)
                ref_x, _ = rm.ffn_forward(x, ww)
                refs = [rm.vad_utterance(u, ww) for u in utts]
                ro = plan.row_offsets
                for it in range(200):
                    labels, logits, _ = plan.vad(pcm, want_logits=True)
                    lo_x = hh.ffn_predict(x)[1]
                    st.synchronize()
                    la, lo = labels.cpu().numpy(), logits.cpu().numpy()
                    for i, (c, feats, rl, rlab) in enumerate(refs):
                        g = lo[ro[i]:ro[i + 1]]
                        assert np.all(np.abs(g - rl) <= LOGIT_ATOL + LOGIT_RTOL * np.abs(rl)), (name, it, i)
                        dec = decisive_rows(rl)
                        assert np.array_equal(la[ro[i]:ro[i + 1]][dec], rlab[dec]), (name, it, i)
                    gx = lo_x.cpu().numpy()
                    assert np.all(np.abs(gx - ref_x) <= LOGIT_ATOL + LOGIT_RTOL * np.abs(ref_x)), (name, it)
            hh.close()
            results[name] = "ok"
        except BaseException as ex:  # noqa: BLE001 -- reported by the main thread
            results[name] = repr(ex)

    ts = [threading.Thread(target=worker, args=("a", 101, "tc16")), threading.Thread(target=worker, args=("b", 202, "fp32")),
          threading.Thread(target=worker, args=("c", 303, "tc"))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert results == {"a": "ok", "b": "ok", "c": "ok"}, results


def test_cfg4_4096_streams_against_offline_labels(hw):
    """configs[3] at the configured size: 4096 concurrent streams, 40 ticks of 10 ms through the CUDA-graph
    tick of StreamBank; every stream's decisions equal the offline fused kernel on the same samples, and
    sampled streams agree with the oracle."""
    from vad_b200 import batch
    from vad_b200.analyser import StreamBank
    h, w = hw
    h.set_ffn_impl("fp32")     # the stream kernel's FFN is FP32: compare with the FP32 offline path bit for bit
    n_streams, n_chunks = 4096, 40
    L = 160 * n_chunks
    utts = [synth_utterance(41, s, L) for s in range(n_streams)]
    allpcm = np.stack(utts)                                                    # [4096, 6400]
    bank = StreamBank(n_streams, handle=h)
    assert bank.use_graph
    got = np.full((n_streams, n_chunks), 255, np.uint8)
    for j in range(n_chunks):
        bank.h_chunks.numpy()[:] = allpcm[:, 160 * j:160 * (j + 1)]
        got[:, j] = bank.feed_pinned().numpy()
    assert bank._graphs, "ticks must replay a captured CUDA graph"
    assert np.all(got[:, :7] == 255) and np.all(got[:, 7:] <= 1)
    off_labels = batch.vad_batch(utts, handle=h)
    k = n_chunks - 7
    offl = np.stack([o.cpu().numpy()[:k] for o in off_labels])
    assert offl.shape == (n_streams, k)
    assert np.array_equal(got[:, 7:], offl)
    for s in (0, 31, 32, 2048, 4095):
        _, _, ref_logits, ref_labels = rm.vad_utterance(utts[s], w)
        dec = decisive_rows(ref_logits[:k])
        assert np.array_equal(got[s, 7:][dec], ref_labels[:k][dec])
    # a second bank on the same handle, plain launches (no graph): same decisions
    bank2 = StreamBank(n_streams, handle=h, use_graph=False)
    for j in range(12):
        lab = bank2.feed(allpcm[:, 160 * j:160 * (j + 1)])
        assert np.array_equal(lab, got[:, j])
    h.set_ffn_impl("tc16")


def test_bit_identical_frames_define_nan_rows(hw):
    """sigma5 == 0 semantics on low-variance audio.  A tone whose period divides the hop makes every frame
    bit-identical: the reference's z = (c - mean5) / std5 is then a rounding artefact (NaN when (5v)/5 == v
    in float64, else +-1); the kernels define it as NaN -> non-speech.  Hum / near-constant audio with
    tiny but non-zero variance must stay finite and match the oracle within the conditioning-aware bound."""
    from vad_b200 import batch, runtime
    h, w = hw
    n = np.arange(16000 * 2)
    tone = np.round(8000 * np.sin(2 * np.pi * 100.0 * n / 16000.0)).astype(np.int16)     # period 160 = hop
    labels, logits = batch.vad_batch([tone], handle=h, want_logits=True)
    la, lo = labels[0].cpu().numpy(), logits[0].cpu().numpy()
    assert np.all(la == 0) and np.all(np.isnan(lo))
    z = rm.analyser_features(rm.mfcc_utterance(tone))[:, :13]
    assert np.all(np.isnan(z) | (np.abs(np.abs(z) - 1.0) < 1e-6))            # the reference's artefact values
    # hum with a slow drift: frames differ, variance is small; features finite and close to the oracle
    rng = np.random.default_rng(8)
    hum = np.round(3000 * np.sin(2 * np.pi * 50.0 * n / 16000.0) * (1 + 0.2 * n / n.size)
                   + rng.integers(-1, 2, n.size)).astype(np.int16)
    flat, off, ln = batch.pack_utterances([hum])
    plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
    _, lo2, fe2 = plan.vad(flat.to(h.device), want_logits=True, want_feats=True)
    c = rm.mfcc_utterance(hum)
    ref_f = rm.analyser_features(c)
    fin = np.isfinite(ref_f)
    fe2 = fe2.cpu().numpy()
    assert np.array_equal(np.isfinite(fe2), fin)
    sig = np.lib.stride_tricks.sliding_window_view(c, 5, axis=0)[: c.shape[0] - 5].std(axis=2)
    tol = 3e-4 + 2e-4 / np.maximum(np.tile(sig, 3), 1e-12)
    assert np.all(np.abs(fe2 - ref_f)[fin] <= tol[fin])


def test_bench_dump_outputs_hold_the_timed_labels(hw, tmp_path):
    """bench.py --dump-outputs saves the timed step's labels of a seeded sample of utterances: the rows a plan over the
    same seeded workload gives for those utterances, within the 64 MB cap; --steps sets the number of timed launches."""
    import json
    import os
    import subprocess
    import sys
    import torch
    from vad_b200 import batch, runtime
    h, w = hw
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    seed, n_utt, L = 77, 14400, 160000                                         # 40 h of 10 s utterances
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                          "--hours-per-gpu", "40", "--seed", str(seed), "--no-e2e", "--no-cpu-baseline",
                          "--no-extra-configs", "--parity-utts", "0", "--dump-outputs", str(tmp_path / "dump")],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["gpu_launches"] == 2 and line["frames_per_step"] == n_utt * 993
    got = np.load(str(tmp_path / "dump" / "labels.npy"))
    utts = np.load(str(tmp_path / "dump" / "utterances.npy"))
    assert got.dtype == np.float32 and utts.dtype == np.float64 and got.nbytes + utts.nbytes <= 64 << 20
    ids = utts.astype(np.int64)
    assert np.array_equal(ids, utts) and np.all(np.diff(ids) > 0) and 0 <= ids[0] and ids[-1] < n_utt
    assert got.shape == (ids.size, 993) and 10000 < ids.size < n_utt                  # a sample, not the whole output
    h.set_ffn_impl("tc16")                                                      # bench.py's default FFN
    off, ln, stride = batch.uniform_layout(n_utt, L)
    pcm = h.synth_pcm(n_utt, L, seed=seed, first_utt=0, utt_stride=stride)
    labels = runtime.Plan(h, off, ln, runtime.MODE_VAD).vad(pcm)[0].view(n_utt, 993)
    assert np.array_equal(got, labels[torch.from_numpy(ids).to(h.device)].float().cpu().numpy())
    for u in (int(ids[0]), int(ids[-1])):
        check_vad(got[np.searchsorted(ids, u)].astype(np.uint8), None, synth_utterance(seed, u, L), w)
