"""GPU: the 16 kHz resampler and the format decoder against the float64 oracle (oracle/ref_resample.py) under the
rounding contract of tests/_resample_bound.py -- every accepted test rate x the signal catalogue x ragged batches, int16
and float32 input, guard bands around every utterance; decode of every format x channel count x byte order; file
ingest of a mix of formats and rates; the batch API at other rates; graph capture of the resample call."""
import ctypes as C
import struct

import numpy as np
import pytest
import torch
from scipy.io import wavfile

from oracle import ref_math as rm, ref_resample as rr

import _signals
import _resample_bound as rb

pytestmark = pytest.mark.gpu

RATES = [8000, 11025, 22050, 24000, 32000, 44100, 48000, 96000]
SENT = 0x5A5A


@pytest.fixture(scope="module")
def h():
    from vad_b200 import runtime
    return runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))


def _batch(rate):
    """Ragged batch at `rate`: lengths 0, 1, a few samples (shorter than one filter span), the catalogue's full-scale,
    tonal, band-limited and near-silent signals, and 10 s of the mixed utterance."""
    cat = _signals.catalogue()
    names = ["clipped_noise", "square_nyquist", "dc_max", "dc_min", "tone_1k", "tone_7900", "lowpass_300_noise",
             "highpass_7k_noise", "lsb_noise", "impulse_train"]
    utts = [np.zeros(0, np.int16), cat["clipped_noise"][:1], cat["square_nyquist"][:5]]
    utts += [cat[n][:3000 + 37 * i] for i, n in enumerate(names)]
    utts.append(np.resize(cat["mixed"], 10 * rate + 3))
    return utts


def _run_checked(h, rate, utts, as_float):
    """Resampler.run on a packed input with sentinels between utterances, into an output full of sentinels."""
    from vad_b200 import runtime
    r = runtime.Resampler(h, rate)
    lens = np.array([len(u) for u in utts], dtype=np.int64)
    offs = np.zeros(len(utts), dtype=np.int64)
    offs[1:] = np.cumsum(lens[:-1] + 13)                 # 13 guard samples, any alignment
    host = np.full(int(offs[-1] + lens[-1] + 13), 12345, dtype=np.int16)
    for u, o in zip(utts, offs):
        host[o:o + len(u)] = u
    d_in = torch.from_numpy(host.astype(np.float32) if as_float else host).cuda()
    out_offs = r.output_offsets(lens)
    out = torch.full((int(out_offs[-1]) + 64,), SENT, dtype=torch.int16, device="cuda")
    pcm, o16, l16 = r.run(d_in, offs, lens, out=out)
    torch.cuda.synchronize()
    assert np.array_equal(o16, out_offs[:-1])
    got = pcm.cpu().numpy()
    outside = np.ones(got.size, dtype=bool)
    total = band = 0
    for u, o, n in zip(utts, o16, l16):
        assert n == rr.resample_exact(u, rate).size
        t, b = rb.check(got[o:o + n], rate, u.astype(np.float64))
        total, band = total + t, band + b
        outside[o:o + n] = False
    assert np.all(got[outside] == SENT), "writes outside the utterances' outputs"
    return total, band


@pytest.mark.parametrize("as_float", [False, True], ids=["int16", "float32"])
@pytest.mark.parametrize("rate", RATES + [16000])
def test_resample_rounding_contract(h, rate, as_float):
    total, band = _run_checked(h, rate, _batch(rate), as_float)
    # the band is empty for near-silent audio and holds a few per cent of full-scale outputs, where the worst-case
    # rounding of up to 481 float32 FMAs reaches 0.1 LSB; those outputs are still held to 1 LSB
    print("rate %d %s: %d outputs, %d in the rounding band" % (rate, "f32" if as_float else "s16", total, band))
    assert band <= total // 4


@pytest.mark.parametrize("rate", [44100, 131072, 4000, 384000])
def test_resample_float_input_and_extreme_ratios(h, rate):
    """Non-integer float input, and the ratios at the ends of the accepted range (longest filter, up 4, down 24)."""
    from vad_b200 import runtime
    rng = np.random.default_rng(rate)
    utts = [rng.standard_normal(n) * 9000.0 for n in (0, 3, 777, 20011)]
    v = [u.astype(np.float32) for u in utts]
    r = runtime.Resampler(h, rate)
    lens = np.array([len(u) for u in v], dtype=np.int64)
    offs = np.concatenate([[0], np.cumsum(lens[:-1])]).astype(np.int64)
    d_in = torch.from_numpy(np.concatenate(v).astype(np.float32)).cuda()
    pcm, o16, l16 = r.run(d_in, offs, lens)
    got = pcm.cpu().numpy()
    for u, f, o, n in zip(utts, v, o16, l16):
        rb.check(got[o:o + n], rate, u, f, np.abs(f.astype(np.float64) - u))


# ---- decode ----------------------------------------------------------------------------------------------------
def _encode(code, vals, be):
    """int16-unit test values -> (file samples, raw bytes) for format `code`."""
    rng = np.random.default_rng(code)
    n = vals.size
    if code == 1:
        s = rng.integers(0, 256, n).astype(np.uint8)
        return s, s.tobytes()
    if code == 0:
        s = vals.astype(np.int16)
        return s, s.astype(">i2" if be else "<i2").tobytes()
    if code == 2:
        s = rng.integers(-2 ** 23, 2 ** 23, n).astype(np.int32)
        b = s.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3]
        return s, (b[:, ::-1] if be else b).tobytes()
    if code == 3:
        s = rng.integers(-2 ** 31, 2 ** 31, n).astype(np.int64).astype(np.int32)
        return s, s.astype(">i4" if be else "<i4").tobytes()
    s = rng.uniform(-1.2, 1.2, n)
    s[::97] = np.nan
    s[5::101] = np.inf
    if code == 4:
        s = s.astype(np.float32)
        return s, s.astype(">f4" if be else "<f4").tobytes()
    return s, s.astype(">f8" if be else "<f8").tobytes()


FMT = {0: "s16", 1: "u8", 2: "s24", 3: "s32", 4: "f32", 5: "f64"}


@pytest.mark.parametrize("be", [False, True], ids=["le", "be"])
@pytest.mark.parametrize("ch", [1, 2, 6])
@pytest.mark.parametrize("code", [0, 1, 2, 3, 4, 5])
def test_decode_pcm(h, code, ch, be):
    n = 5003
    s, raw = _encode(code, np.random.default_rng(7).integers(-32768, 32768, n * ch), be)
    bps = {0: 2, 1: 1, 2: 3, 3: 4, 4: 4, 5: 8}[code]
    d_raw = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda()
    # three segments, the last a gap-free tail; destinations with guards between them
    src, ln = [0, 1000, 4000], [700, 2500, 1003]
    dst = [0, 800, 3400]
    out = torch.full((4500,), -7.0, dtype=torch.float32, device="cuda")
    h.decode_pcm(d_raw, code, ch, src, dst, ln, out, big_endian=be)
    got = out.cpu().numpy()
    v = rr.to_units(s, FMT[code]).reshape(n, ch)
    want = rr.downmix(v)
    exact = code in (0, 1, 2, 4)
    delta = rb.decode_delta(v, ch, exact)
    mask = np.ones(got.size, dtype=bool)
    for a, b, k in zip(src, dst, ln):
        g, w, d = got[b:b + k].astype(np.float64), want[a:a + k], delta[a:a + k]
        if exact and ch == 1:
            assert np.array_equal(g, w)
        else:
            assert np.all(np.abs(g - w) <= d), np.max(np.abs(g - w) - d)
        mask[b:b + k] = False
    assert np.all(got[mask] == -7.0)
    assert bps * ch * n == len(raw)


# ---- file ingest -----------------------------------------------------------------------------------------------
def _wav(path, rate, ch, bits, tag, payload):
    ba = ch * bits // 8
    fmt = struct.pack("<HHIIHH", tag, ch, rate, rate * ba, ba, bits)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(payload)) + payload
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def test_device_ingest_resample_mix(h, tmp_path):
    from vad_b200 import batch, io, runtime
    cat = _signals.catalogue()
    rng = np.random.default_rng(11)
    files = []
    # 8 kHz stereo u8
    u8 = rng.integers(0, 256, (8000 * 2 + 77, 2)).astype(np.uint8)
    p = str(tmp_path / "a.wav"); wavfile.write(p, 8000, u8); files.append((p, None, 8000, rr.downmix(rr.to_units(u8, "u8")), None))
    # 44.1 kHz mono s24
    s24 = (np.resize(cat["mixed"], 44100 + 501).astype(np.int32) << 8) + rng.integers(0, 256, 44100 + 501)
    b = s24.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes()
    p = str(tmp_path / "b.wav"); _wav(p, 44100, 1, 24, 1, b); files.append((p, None, 44100, rr.to_units(s24, "s24"), None))
    # 48 kHz stereo f32 with a .stm
    f32 = (rng.standard_normal((48000 * 3, 2)) * 0.3).astype(np.float32)
    p = str(tmp_path / "c.wav"); wavfile.write(p, 48000, f32)
    stm = str(tmp_path / "c.stm")
    with open(stm, "w") as f:
        f.write("c 1 spk 0.25 1.1 <o,f0,male> hello there\n")
        f.write("c 1 spk 1.3 1.31 <o,f0,male> x\n")
        f.write("c 1 spk 1.5 2.75 <o,f0,male> and more words\n")
    s, e = io.parse_stm(stm, 48000)
    mono = rr.downmix(rr.to_units(f32, "f32"))
    stm_x = np.concatenate([mono[a:bb] for a, bb in zip(s, e)])
    vf = np.concatenate([(f32[a:bb].astype(np.float32).sum(axis=1, dtype=np.float32) / np.float32(2)) * 32768
                         for a, bb in zip(s, e)])
    files.append((p, stm, 48000, stm_x, vf))
    # 16 kHz mono s16
    s16 = cat["clipped_noise"]
    p = str(tmp_path / "d.wav"); wavfile.write(p, 16000, s16); files.append((p, None, 16000, s16.astype(np.float64), None))

    ing = io.DeviceIngest(h, resample=True)
    for p, t, _, _, _ in files:
        ing.add(p, t)
    d_pcm, offs, lens, rates = ing.run()
    torch.cuda.synchronize()
    assert rates == [16000] * 4
    got = d_pcm.cpu().numpy()
    for (p, t, rate, x, vf), o, n in zip(files, offs, lens):
        g = got[o:o + n]
        if rate == 16000:
            assert np.array_equal(g, x.astype(np.int16))
        elif vf is None:
            rb.check(g, rate, x, None, rb.decode_delta(x if rate != 8000 else rr.to_units(u8, "u8"), 1 if rate != 8000 else 2,
                                                       True))
        else:
            rb.check(g, rate, x, vf, rb.decode_delta(rr.to_units(np.concatenate([f32[a:bb] for a, bb in zip(s, e)]), "f32"),
                                                     2, True))
    # MODE_DATASET rows of the ingested batch == mfcc_batch on its int16
    plan = runtime.Plan(h, offs, lens, runtime.MODE_DATASET)
    rows = plan.mfcc(d_pcm).cpu().numpy()
    ref = batch.mfcc_batch([got[o:o + n] for o, n in zip(offs, lens)], deltas=True, handle=h)
    for u in range(4):
        assert np.array_equal(rows[plan.row_offsets[u]:plan.row_offsets[u + 1]], ref[u].cpu().numpy())
    # the 16 kHz s16 file: bit-identical to the path without resampling
    plain = io.DeviceIngest(h)
    plain.add(files[3][0])
    p_pcm, p_offs, p_lens, _ = plain.run()
    rows_plain = runtime.Plan(h, p_offs, p_lens, runtime.MODE_DATASET).mfcc(p_pcm).cpu().numpy()
    assert np.array_equal(rows[plan.row_offsets[3]:plan.row_offsets[4]], rows_plain)


# ---- batch API at other rates ----------------------------------------------------------------------------------
@pytest.mark.parametrize("rate", [8000, 44100, 48000])
def test_batch_api_at_other_rates(h, rate):
    from vad_b200 import batch
    rng = np.random.default_rng(rate)
    cat = _signals.catalogue()
    utts = [np.resize(cat["mixed"], rate * 2 + 19), np.resize(cat["tone_1k"], rate + 5),
            (rng.standard_normal(rate * 3) * 6000).astype(np.int16)]
    res = batch.resample(utts, rate, handle=h)
    for u, r16 in zip(utts, res):
        rb.check(r16, rate, u.astype(np.float64))
    lab = batch.vad_batch(utts, handle=h, sample_rate=rate)
    ref = batch.vad_batch(res, handle=h)
    for a, b in zip(lab, ref):
        assert np.array_equal(a.cpu().numpy(), b.cpu().numpy())
    mf = batch.mfcc_batch(utts, handle=h, sample_rate=rate)
    mref = batch.mfcc_batch(res, handle=h)
    for a, b in zip(mf, mref):
        assert np.array_equal(a.cpu().numpy(), b.cpu().numpy())
    segs = batch.speech_segments(utts, handle=h, sample_rate=rate, min_silence_ms=50)
    s16 = batch.speech_segments(res, handle=h, min_silence_ms=50)
    up, down = rr.ratio(rate)
    for sg, s, u in zip(segs, s16, utts):
        assert sg.shape == s.shape
        assert np.array_equal(sg[:, 0], s[:, 0] * down // up)
        assert np.array_equal(sg[:, 1], np.minimum(len(u), -((-s[:, 1] * down) // up)))
        assert np.all(sg[:, 0] < sg[:, 1])
    sp = batch.extract_speech(utts, handle=h, sample_rate=rate, min_silence_ms=50)
    sp16 = batch.extract_speech(res, handle=h, min_silence_ms=50)
    for a, b in zip(sp, sp16):
        assert np.array_equal(a, b)
    # float input in [-1, 1]: scaled by 32768 on the device
    fl = [u.astype(np.float32) / 32768.0 for u in utts]
    for a, b in zip(batch.resample(fl, rate, handle=h), res):
        assert np.array_equal(a, b)


def test_resample_packed_in_a_cuda_graph(h):
    from vad_b200 import runtime
    from vad_b200.runtime import _ptr
    rate = 44100
    r = runtime.Resampler(h, rate)
    utts = _batch(rate)[:8]
    lens = np.array([len(u) for u in utts], dtype=np.int64)
    offs = np.concatenate([[0], np.cumsum(lens[:-1])]).astype(np.int64)
    d_in = torch.from_numpy(np.concatenate(utts)).cuda()
    ref, o16, l16 = r.run(d_in, offs, lens)
    torch.cuda.synchronize()
    out_offs = np.zeros(len(utts) + 1, dtype=np.int64)
    ws_bytes = int(h.lib.vadb200_resample_workspace_bytes(r._r, len(utts)))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    out = torch.zeros_like(ref)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            cs = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            assert h.lib.vadb200_resample_packed(r._r, runtime.PCM_S16, _ptr(d_in), offs.ctypes.data_as(C.c_void_p),
                                                 lens.ctypes.data_as(C.c_void_p), len(utts), _ptr(out), out.numel(),
                                                 out_offs.ctypes.data_as(C.c_void_p), _ptr(ws), ws_bytes, cs) == 0
    out.fill_(0)
    ws.fill_(0)
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(out_offs[:-1], o16)
    assert np.array_equal(out.cpu().numpy(), ref.cpu().numpy())
    g.reset()
