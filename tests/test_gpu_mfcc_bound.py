"""GPU: every MFCC row and window feature, entry by entry, on the kernel's own float32 inputs.

* get_spec_mag (frames_kernel) equals the host replay of vad_core.cuh's FFT (tests/_mfcc_bound.py power_f32) bit for
  bit, on int16-valued and non-integer frames of 400, 399, 1 and 512 samples, with no front end and with pre-emphasis
  0.97 (+ Hamming on the 400-sample frames: a window needs them).
* MFCC rows are within tests/_mfcc_bound.py's bound of the replayed powers: fused MODE 0 (plan MFCC, automatic and
  fixed segment lengths, identical bits across them), the host pipeline, get_mfcc (frames_kernel) and
  get_mfcc_from_spec (spec_to_mfcc_kernel) on the caller's exact spectra.
* Dataset rows (MODE 1) equal MODE 0's rows and their fp32 differences bit for bit.
* VAD features (want_feats) under fp32, tc and tc16, and vad_windows, follow tests/_window_bound.py's rules on the
  MODE 0 rows of the same handle: d1 bit-exact (so the VAD kernel's MFCC ring holds the bits MODE 0 writes), the
  analyser z and d2 within the bound, NaN exactly where the rule puts it -- bit-identical windows on the packed path
  (window_features_pairs: tc, tc16, dataset rows), ==-equal ones on the scalar path (window_features through
  classify_row: the fp32 block phase and windows_kernel).  The features are identical across the three FFN paths.

Front ends: none, pre-emphasis 0.97 + Hamming, and pre-emphasis 1 with a window holding zeros.  Utterances: the
signal catalogue, digital silence, DC, a +-32767 square at Nyquist, a single impulse, bin-centred tones, and a
ragged batch whose utterances end at every residue of the 32-frame step and at 32 block-phase positions."""
import numpy as np
import pytest

from oracle import ref_math as rm

import _mfcc_bound as mb
import _signals
import _window_bound as wb

pytestmark = pytest.mark.gpu

SEGMENT_FRAMES = (0, 64, 128, 160, 2048)
HAMMING = np.hamming(400)
ZERO_WINDOW = np.hamming(400) * (np.arange(400) % 7 != 3)
ZERO_WINDOW[:24] = 0
ZERO_WINDOW[-17:] = 0
FRONT_ENDS = {"default": None, "a0.97_hamming": (0.97, HAMMING), "a1_zeros": (1.0, ZERO_WINDOW)}
WORST = {}


def samples_for_frames(T):
    return rm.FRAME_SIZE + (T - 1) * rm.FRAME_STEP + 1


def utterances():
    out = list(_signals.catalogue().values())
    n = 16000
    t = np.arange(n)
    out += [np.zeros(n, np.int16), np.full(n, 1234, np.int16),
            np.where(t % 2 == 0, 32767, -32767).astype(np.int16)]
    imp = np.zeros(n, np.int16)
    imp[5003] = 32767
    out.append(imp)
    for k in (20, 64, 200):                 # bin-centred: frequency k 16000 / 512, one mel band lit, the rest noise
        out.append(np.round(20000 * np.sin(2 * np.pi * k * t / 512.0)).astype(np.int16))
    for i in range(32):                      # T = 270 + 33 i: every residue mod 32, 32 positions mod 256
        out.append(_signals.clipped_noise(samples_for_frames(270 + 33 * i), seed=100 + i) // 3)
    return [np.ascontiguousarray(u, np.int16) for u in out]


UTTS = utterances()
_POWER = {}


def power(i, fe_name):
    if (i, fe_name) not in _POWER:
        _POWER[(i, fe_name)] = mb.power_pcm(UTTS[i], FRONT_ENDS[fe_name])
    return _POWER[(i, fe_name)]


def note(key, frac):
    WORST[key] = max(WORST.get(key, 0.0), frac)


def check_mfcc(entry, C, P):
    ref, bnd, _ = mb.mfcc_bound(np.nan_to_num(P))
    C = np.asarray(C, np.float32)
    assert C.shape == ref.shape, (entry, C.shape, ref.shape)
    err = np.abs(C.astype(np.float64) - ref)
    bad = ~(err <= bnd)
    assert not bad.any(), "%s: %d entries exceed the bound (worst |d| / bound %.3g, rows %s)" % (
        entry, bad.sum(), np.max(err / bnd), np.unique(np.nonzero(bad)[0])[:10].tolist())
    note(("MFCC", entry), float(np.max(err / bnd)))


@pytest.fixture(scope="module")
def handle():
    import torch
    from vad_b200 import runtime
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    h = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    yield h
    h.close()
    if WORST:
        print("\nworst |d| / bound:")
        for k in sorted(WORST):
            print("  %-6s %-40s %.4f" % (k[0], k[1], WORST[k]))


def set_fe(h, fe):
    h.set_frontend(0.0, None) if fe is None else h.set_frontend(fe[0], fe[1])


def test_spec_frames_equal_replay(handle):
    rng = np.random.default_rng(7)
    try:
        for fe_name in ("default", "a0.97_hamming"):
            for n in (400, 399, 1, 512):
                fe = FRONT_ENDS[fe_name]
                if fe is not None and n != 400:      # a window needs 400-sample frames: pre-emphasis alone
                    fe = (fe[0], None)
                set_fe(handle, fe)
                for kind in ("int16", "real"):
                    fr = rng.integers(-32768, 32768, (37, n)).astype(np.float32) if kind == "int16" else \
                        (rng.standard_normal((37, n)) * 1234.567).astype(np.float32)
                    got = handle.spec_frames(fr).cpu().numpy()
                    want = mb.spec_f32(fr, fe)
                    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (fe_name, n, kind)
                    check_mfcc("get_mfcc %s" % fe_name, handle.mfcc_frames(fr).cpu().numpy(), mb.power_f32(fr, fe))
    finally:
        set_fe(handle, None)


def test_mfcc_from_spec_within_bound(handle):
    rng = np.random.default_rng(8)
    fr = rm.split_into_frames(UTTS[0])[:64].astype(np.float32)
    spec = mb.spec_f32(fr)
    cases = [spec]
    z = spec.copy()
    z[:, 40:60] = 0                                          # zero bins inside several triangles
    z[::5, 12:14] = 0
    cases.append(z)
    cases.append(np.zeros((33, 256), np.float32))            # all-zero frames: every filter takes the eps branch
    huge = np.float32(2.0 ** -20 * (65536.0 * 400) ** 2)
    cases.append((huge * rng.uniform(0.5, 1.0, (40, 256))).astype(np.float32))
    cases.append((np.float32(1e-30) * rng.uniform(0, 1, (40, 256))).astype(np.float32))   # tiny bins
    one = np.zeros((5, 256), np.float32)
    one[np.arange(5), [10, 50, 128, 200, 255]] = 3.0         # one bin per frame: one or two filters non-zero
    cases.append(one)
    for s in cases:
        got = handle.mfcc_from_spec(s).cpu().numpy()
        check_mfcc("get_mfcc_from_spec", got, s * np.float32(2.0 ** 20))


@pytest.mark.parametrize("fe_name", list(FRONT_ENDS))
def test_fused_mfcc_rows_within_bound(handle, fe_name):
    import torch
    from vad_b200 import batch, runtime
    fe = FRONT_ENDS[fe_name]
    set_fe(handle, fe)
    flat, off, ln = batch.pack_utterances(UTTS)
    pcm = flat.to(handle.device)
    try:
        first = None
        for sf in SEGMENT_FRAMES:
            handle.set_plan_segment_frames(sf)
            plan = runtime.Plan(handle, off, ln, runtime.MODE_MFCC)
            rows = plan.mfcc(pcm).cpu().numpy()
            if first is None:
                first = rows
                ro = plan.row_offsets
                for i in range(len(UTTS)):
                    check_mfcc("fused MODE 0 %s" % fe_name, rows[ro[i]:ro[i + 1]], power(i, fe_name))
                host = plan.mfcc_host(flat).numpy()
                assert np.array_equal(host.view(np.uint32), rows.view(np.uint32)), "host pipeline"
            else:
                assert np.array_equal(rows.view(np.uint32), first.view(np.uint32)), sf
            plan.close()
        # dataset rows: MODE 0's c and its fp32 differences, bit for bit
        handle.set_plan_segment_frames(0)
        plan = runtime.Plan(handle, off, ln, runtime.MODE_DATASET)
        ds = plan.mfcc(pcm).cpu().numpy()
        torch.cuda.synchronize()
        mro = runtime.Plan(handle, off, ln, runtime.MODE_MFCC).row_offsets
        for i in range(len(UTTS)):
            wb.window_check(first[mro[i]:mro[i + 1]], ds[plan.row_offsets[i]:plan.row_offsets[i + 1]], "dataset",
                            "pairs")
        plan.close()
    finally:
        handle.set_plan_segment_frames(0)
        set_fe(handle, None)


@pytest.mark.parametrize("fe_name", ["default", "a0.97_hamming"])
def test_vad_features_follow_window_rules(handle, fe_name):
    import torch
    from vad_b200 import batch, runtime
    fe = FRONT_ENDS[fe_name]
    set_fe(handle, fe)
    flat, off, ln = batch.pack_utterances(UTTS)
    pcm = flat.to(handle.device)
    try:
        mplan = runtime.Plan(handle, off, ln, runtime.MODE_MFCC)
        c = mplan.mfcc(pcm).cpu().numpy()
        mro = mplan.row_offsets
        mfcc = [c[mro[i]:mro[i + 1]] for i in range(len(UTTS))]
        for sf in (0, 160):
            handle.set_plan_segment_frames(sf)
            plan = runtime.Plan(handle, off, ln, runtime.MODE_VAD)
            ro = plan.row_offsets
            for fm, mode in ((runtime.FEAT_ANALYSER, "analyser"), (runtime.FEAT_DATASET, "dataset")):
                per = {}
                for impl in ("fp32", "tc", "tc16"):
                    handle.set_ffn_impl(impl)
                    _, _, feats = plan.vad(pcm, want_feats=True, feat_mode=fm)
                    torch.cuda.synchronize()
                    feats = feats.cpu().numpy()
                    path = "scalar" if impl == "fp32" else "pairs"
                    for i in range(len(UTTS)):
                        r = wb.window_check(mfcc[i], feats[ro[i]:ro[i + 1]], mode, path)
                        for k, v in r.items():
                            note((k, "fused VAD %s %s" % (impl, fe_name)), v)
                    per[impl] = feats
                for impl in ("tc", "tc16"):
                    same = (per[impl].view(np.uint32) == per["fp32"].view(np.uint32)) | \
                        (np.isnan(per[impl]) & np.isnan(per["fp32"]))
                    assert same.all(), (impl, mode, int((~same).sum()))
            plan.close()
        # vad_windows (windows_kernel, classify_row) on the same rows
        win = np.concatenate([wb.windows(m) for m in mfcc])
        for fm, mode in ((runtime.FEAT_ANALYSER, "analyser"), (runtime.FEAT_DATASET, "dataset")):
            _, _, feats = handle.vad_windows(np.ascontiguousarray(win), feat_mode=fm, want_feats=True)
            feats = feats.cpu().numpy()
            o = 0
            for m in mfcc:
                n = m.shape[0] - 5
                r = wb.window_check(m, feats[o:o + n], mode, "scalar")
                for k, v in r.items():
                    note((k, "vad_windows %s" % fe_name), v)
                o += n
        mplan.close()
    finally:
        handle.set_plan_segment_frames(0)
        handle.set_ffn_impl("tc16")
        set_fe(handle, None)
