"""GPU: lifetime and error paths of the C ABI's objects (handle, plan, stream bank, trainer), and the number of kernel
launches each entry point adds to vadb200_launch_count, called through vad_b200._lib."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import ref_math as rm

pytestmark = pytest.mark.gpu

E_CUDA = -3
MODE_MFCC, MODE_DATASET, MODE_VAD = 0, 1, 2
FFN_KEYS = ("W1", "b1", "W2", "b2", "W3", "b3", "W4", "b4")


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


@pytest.fixture(scope="module")
def lib():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vad_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def h(lib):
    from vad_b200 import runtime
    hd = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    yield hd
    hd.close()


@pytest.fixture(scope="module")
def utts(golden_dir):
    """The golden utterances packed at 8-sample-aligned offsets: (offsets, lengths, host int16 PCM)."""
    z = np.load(os.path.join(golden_dir, "utterances.npz"))
    pcms = [z[n + "/pcm"] for n in sorted({k.split("/")[0] for k in z.files})]
    lens = np.array([len(p) for p in pcms], np.int64)
    offs = np.zeros_like(lens)
    offs[1:] = np.cumsum((lens[:-1] + 7) // 8 * 8)
    pcm = np.zeros(int(offs[-1] + lens[-1]) + 8, np.int16)
    for o, p in zip(offs, pcms):
        pcm[o:o + len(p)] = p
    return offs, lens, pcm


def create_plan(lib, handle_ptr, offs, lens, mode):
    p = C.c_void_p()
    offs = np.ascontiguousarray(offs, np.int64)
    lens = np.ascontiguousarray(lens, np.int64)
    assert lib.vadb200_plan_create(handle_ptr, offs.ctypes.data_as(C.c_void_p), lens.ctypes.data_as(C.c_void_p),
                                   len(offs), mode, C.byref(p)) == 0, lib.vadb200_last_error()
    return p


def test_failed_creates_leave_null_and_no_stale_error(lib, h, utts):
    import torch
    offs, lens, pcm_h = utts
    plan = create_plan(lib, h._h, offs, lens, MODE_VAD)
    try:
        rows = int(lib.vadb200_plan_total_rows(plan))
        pcm = torch.from_numpy(pcm_h).cuda()
        before = torch.empty(rows, dtype=torch.uint8, device="cuda")
        after = torch.full((rows,), 255, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        assert lib.vadb200_vad_packed(plan, _ptr(pcm), pcm.numel(), _ptr(before), None, None, 0, None) == 0
        torch.cuda.synchronize()

        # requests no B200 can satisfy: 687 GB of stream history, ~180 TB of trainer partials.  Each is one
        # cudaErrorMemoryAllocation, which leaves the context usable.
        b = C.c_void_p(1)
        assert lib.vadb200_stream_bank_create(h._h, 2 ** 30, C.byref(b)) == E_CUDA
        assert not b.value
        t = C.c_void_p(1)
        assert lib.vadb200_trainer_create(h._h, 2 ** 40, 1.0, 0.95, 1e-8, C.byref(t)) == E_CUDA
        assert not t.value

        # the same thread, no other CUDA call in between: the next launch reports only itself
        rc = lib.vadb200_vad_packed(plan, _ptr(pcm), pcm.numel(), _ptr(after), None, None, 0, None)
        assert rc == 0, lib.vadb200_last_error()
        torch.cuda.synchronize()
        assert torch.equal(before, after)
    finally:
        lib.vadb200_plan_destroy(plan)


def launches(lib, fn):
    import torch
    torch.cuda.synchronize()
    n0 = lib.vadb200_launch_count()
    fn()
    torch.cuda.synchronize()
    return lib.vadb200_launch_count() - n0


def test_launch_count_per_entry_point(lib, h, utts):
    import torch
    from vad_b200 import runtime
    offs, lens, pcm_h = utts
    pcm = torch.from_numpy(pcm_h).cuda()
    dev = pcm.device
    pl = {m: runtime.Plan(h, offs, lens, m) for m in (MODE_MFCC, MODE_DATASET, MODE_VAD)}
    rng = np.random.default_rng(0)
    frames = torch.from_numpy(rng.standard_normal((40, 400)).astype(np.float32)).cuda()
    spec = torch.from_numpy(rng.random((40, 256)).astype(np.float32)).cuda()
    rows39 = torch.from_numpy(rng.standard_normal((300, 39)).astype(np.float32)).cuda()
    windows = torch.from_numpy(rng.standard_normal((50, 5, 13)).astype(np.float32)).cuda()
    labels, _, _ = pl[MODE_VAD].vad(pcm)
    assert launches(lib, lambda: pl[MODE_MFCC].mfcc(pcm)) == 1
    assert launches(lib, lambda: pl[MODE_DATASET].mfcc(pcm)) == 1
    assert launches(lib, lambda: pl[MODE_VAD].vad(pcm)) == 1
    assert launches(lib, lambda: h.spec_frames(frames)) == 1
    assert launches(lib, lambda: h.mfcc_frames(frames)) == 1
    assert launches(lib, lambda: h.mfcc_from_spec(spec)) == 1
    assert launches(lib, lambda: h.vad_windows(windows)) == 1
    assert launches(lib, lambda: h.ffn_predict(rows39)) == 1
    assert launches(lib, lambda: h.get_deltas(rows39, rows39)) == 1
    assert launches(lib, lambda: h.lifter(rows39[:, :13].contiguous())) == 1
    assert launches(lib, lambda: h.scale_rows(rows39.clone())) == 3
    raw = torch.from_numpy(pcm_h.view(np.uint8).copy()).cuda()
    dst = torch.zeros(4096, dtype=torch.int16, device=dev)
    assert launches(lib, lambda: h.ingest_pcm(raw, [0, 1000], [0, 2000], [1000, 2000], dst)) == 1
    assert launches(lib, lambda: h.synth_pcm(3, 1600)) == 1
    assert launches(lib, lambda: h.fp32_peak(0, iters=16)) == 5

    # host path: one fused launch per chunk of whole utterances
    pcm_pin = torch.from_numpy(pcm_h).pin_memory()
    assert launches(lib, lambda: pl[MODE_VAD].vad_host(pcm_pin)) == 1
    long_utts = lens > 4096
    plan_long = runtime.Plan(h, offs[long_utts], lens[long_utts], MODE_VAD)
    h.set_host_chunk_samples(4096)
    try:
        assert launches(lib, lambda: plan_long.vad_host(pcm_pin)) == int(long_utts.sum())
    finally:
        h.set_host_chunk_samples(32 << 20)

    # speech segments: smooth + scan + segments, without the smooth pass when the plan has no tiles
    res = {}
    assert launches(lib, lambda: res.update(seg=pl[MODE_VAD].speech_segments(labels, 100, 100, 30))) == 3
    segs, so, sp, _ = res["seg"]
    assert launches(lib, lambda: pl[MODE_VAD].gather_speech(pcm, segs, so, sp)) == 1
    no_rows = runtime.Plan(h, [0], [1041], MODE_VAD)
    assert no_rows.total_rows == 0
    empty = torch.empty(0, dtype=torch.uint8, device=dev)
    assert launches(lib, lambda: no_rows.speech_segments(empty)) == 2

    # stream bank
    bank = runtime.StreamBankHandle(h, 64)
    chunks = torch.zeros((64, 160), dtype=torch.int16, device=dev)
    lab = torch.empty(64, dtype=torch.uint8, device=dev)
    assert launches(lib, lambda: bank.feed_ptr(chunks.data_ptr(), lab.data_ptr())) == 1
    bank.set_speech(3, 3, 3)
    srows = torch.empty(64, dtype=torch.uint8, device=dev)
    bounds = torch.empty(64, dtype=torch.int64, device=dev)
    assert launches(lib, lambda: bank.feed_speech_ptr(chunks.data_ptr(), lab.data_ptr(), 0, srows.data_ptr(),
                                                      bounds.data_ptr())) == 1
    end = torch.ones(64, dtype=torch.uint8, device=dev)
    tail_rows = torch.empty((64, bank.speech_delay() + 1), dtype=torch.uint8, device=dev)
    tail_bounds = torch.empty((64, 2 * bank.speech_delay() + 2), dtype=torch.int64, device=dev)
    assert launches(lib, lambda: bank.end_streams_ptr(end.data_ptr(), tail_rows.data_ptr(),
                                                      tail_bounds.data_ptr())) == 1
    bank.close()

    # training step: gradient + update
    from vad_b200.trainer import FFNTrainer
    tr = FFNTrainer(h, rm.glorot_ffn(1), max_batch=512)
    y = torch.from_numpy(rng.integers(0, 3, 300).astype(np.uint8)).cuda()
    assert launches(lib, lambda: tr.train_on_batch(rows39, y)) == 2
    tr.close()
    for p in list(pl.values()) + [plan_long, no_rows]:
        p.close()


def test_destroy_handle_before_its_objects(lib, utts):
    import torch
    from vad_b200 import _lib
    offs, lens, _ = utts
    cfg = _lib.Config()
    lib.vadb200_default_config(C.byref(cfg))
    hd = C.c_void_p()
    assert lib.vadb200_create(C.byref(cfg), 0, C.byref(hd)) == 0, lib.vadb200_last_error()
    w = rm.glorot_ffn(2)
    arrs = [np.ascontiguousarray(w[k], np.float32) for k in FFN_KEYS]
    assert lib.vadb200_set_ffn_weights(hd, *[a.ctypes.data_as(C.c_void_p) for a in arrs]) == 0
    plan = create_plan(lib, hd, offs, lens, MODE_VAD)
    bank, tr = C.c_void_p(), C.c_void_p()
    assert lib.vadb200_stream_bank_create(hd, 8, C.byref(bank)) == 0, lib.vadb200_last_error()
    assert lib.vadb200_stream_bank_set_speech(bank, 1, 3, 3, 3, None) == 0, lib.vadb200_last_error()
    assert lib.vadb200_trainer_create(hd, 1000, 1.0, 0.95, 1e-8, C.byref(tr)) == 0, lib.vadb200_last_error()
    torch.cuda.synchronize()

    assert lib.vadb200_destroy(hd) == 0
    assert lib.vadb200_plan_destroy(plan) == 0
    assert lib.vadb200_stream_bank_destroy(bank) == 0
    assert lib.vadb200_trainer_destroy(tr) == 0
    for destroy in (lib.vadb200_destroy, lib.vadb200_plan_destroy, lib.vadb200_stream_bank_destroy,
                    lib.vadb200_trainer_destroy):
        assert destroy(None) == 0
    torch.cuda.synchronize()  # the frees left no error behind on the device
