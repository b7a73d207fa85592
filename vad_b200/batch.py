"""Batched / ragged entry points around the fused kernels, plus drop-ins for the reference's offline flow:
``split_into_frames`` / ``process_file`` (dataset/file_processing.py:14-103), ``scale_features``
(dataset/utils.py:5-32), ``process_files`` (dataset_creator.py:19-73) and the feature sink
(file_processing.py:110-148).  Host code only parses containers, packs buffers and shapes results; decode,
segment gather, MFCC / delta rows and the scaling statistics all run on the device."""
import json
import os

import numpy as np
import torch

from . import config, runtime
from .io import ALIGN, DeviceIngest, parse_stm
from .runtime import MODE_MFCC, MODE_DATASET, MODE_VAD, FEAT_ANALYSER, FEAT_DATASET  # noqa: F401


def pack_utterances(utterances, pin=False):
    """List of 1-D int16 arrays -> (flat int16 CPU tensor, offsets int64[n], lengths int64[n]).
    Each utterance starts at a multiple of 8 samples; the tail of the buffer is padded too.
    Replaces the per-file pickling of dataset_creator.process_files (dataset_creator.py:53-65)."""
    lengths = np.array([len(u) for u in utterances], dtype=np.int64)
    padded = (lengths + ALIGN - 1) // ALIGN * ALIGN
    offsets = np.zeros(len(utterances), dtype=np.int64)
    if len(utterances) > 1:
        offsets[1:] = np.cumsum(padded[:-1])
    total = int(padded.sum()) + ALIGN
    flat = torch.zeros(total, dtype=torch.int16)
    if pin:
        flat = flat.pin_memory()
    buf = flat.numpy()
    for u, o, n in zip(utterances, offsets, lengths):
        a = np.asarray(u)
        if a.dtype != np.int16:
            raise TypeError("utterances must be int16 PCM")
        buf[o:o + n] = a
    return flat, offsets, lengths


def uniform_layout(n_utt, utt_samples):
    stride = (utt_samples + ALIGN - 1) // ALIGN * ALIGN
    offsets = np.arange(n_utt, dtype=np.int64) * stride
    lengths = np.full(n_utt, utt_samples, dtype=np.int64)
    return offsets, lengths, stride


def _upload_16k(utterances, handle, sample_rate):
    """One upload of the batch and, at any rate but 16 kHz, the device resampler -> (int16 CUDA tensor, offsets,
    lengths) at 16 kHz.  At 16000 Hz this is pack_utterances and one copy, as before."""
    if int(sample_rate) == config.SAMPLERATE:
        flat, offsets, lengths = pack_utterances(utterances)
        return flat.to(handle.device), offsets, lengths
    return _resample_device(utterances, handle, int(sample_rate))


def _resample_device(utterances, handle, sample_rate):
    r = runtime.Resampler(handle, sample_rate)
    arrs = [np.asarray(u) for u in utterances]
    if all(a.dtype == np.int16 for a in arrs):
        flat, offsets, lengths = pack_utterances(arrs)
        return r.run(flat.to(handle.device), offsets, lengths)
    if not all(a.dtype.kind == "f" for a in arrs):
        raise TypeError("utterances must all be int16 PCM or all floating point in [-1, 1]")
    wide = any(a.dtype.itemsize > 4 for a in arrs)
    dt, fmt = (np.float64, runtime.PCM_F64) if wide else (np.float32, runtime.PCM_F32)
    lengths = np.array([a.size for a in arrs], dtype=np.int64)
    offsets = np.zeros(len(arrs), dtype=np.int64)
    if len(arrs) > 1:
        offsets[1:] = np.cumsum(lengths[:-1])
    host = np.zeros(max(int(lengths.sum()), 1), dtype=dt)
    for a, o, n in zip(arrs, offsets, lengths):
        host[o:o + n] = a.reshape(-1)
    raw = torch.from_numpy(host.view(np.uint8)).to(handle.device)
    f32 = torch.empty(host.size, dtype=torch.float32, device=handle.device)
    keep = lengths > 0                    # decode scales by 32768 on the device, non-finite samples become 0
    for lo in range(0, int(keep.sum()), 65535):
        sl = slice(lo, lo + 65535)
        handle.decode_pcm(raw, fmt, 1, offsets[keep][sl], offsets[keep][sl], lengths[keep][sl], f32)
    return r.run(f32, offsets, lengths)


def resample(utterances, sample_rate, handle=None):
    """Utterances at ``sample_rate`` -> list of int16 arrays at 16 kHz: scipy.signal.resample_poly's filter on the
    device, rounded half to even and saturated (include/vadb200.h).  Input is int16 PCM, or floating point in [-1, 1]
    (the soundfile / torchaudio convention), scaled by 32768 on the device."""
    handle = handle or runtime.default_handle()
    pcm, offsets, lengths = _resample_device(utterances, handle, int(sample_rate))
    host = pcm.cpu().numpy()
    return [host[o:o + n].copy() for o, n in zip(offsets, lengths)]


def _split_rows(t, row_offsets):
    return [t[int(row_offsets[i]):int(row_offsets[i + 1])] for i in range(len(row_offsets) - 1)]


def mfcc_batch(utterances, deltas=False, handle=None, sample_rate=16000):
    """MFCC of every frame of every utterance.  deltas=False -> list of [T_u, 13] tensors;
    deltas=True -> list of [T_u - 5, 39] rows [c, d1, d2] (process_file's output).  At any other ``sample_rate`` the
    batch is resampled to 16 kHz on the device first (``resample``); rows keep the 16 kHz framing."""
    handle = handle or runtime.default_handle()
    pcm, offsets, lengths = _upload_16k(utterances, handle, sample_rate)
    plan = runtime.Plan(handle, offsets, lengths, MODE_DATASET if deltas else MODE_MFCC)
    out = plan.mfcc(pcm)
    return _split_rows(out, plan.row_offsets)


def vad_batch(utterances, handle=None, want_logits=False, feat_mode=FEAT_ANALYSER, sample_rate=16000):
    """Per-frame speech / non-speech labels (uint8) for every utterance; optionally logits.  At any other
    ``sample_rate`` the batch is resampled to 16 kHz on the device first; labels keep the 16 kHz framing."""
    handle = handle or runtime.default_handle()
    if not handle.has_classifier:
        raise RuntimeError("set FFN weights first (Handle.set_ffn_weights)")
    pcm, offsets, lengths = _upload_16k(utterances, handle, sample_rate)
    plan = runtime.Plan(handle, offsets, lengths, MODE_VAD)
    labels, logits, _ = plan.vad(pcm, want_logits=want_logits, feat_mode=feat_mode)
    lab = _split_rows(labels, plan.row_offsets)
    if want_logits:
        return lab, _split_rows(logits, plan.row_offsets)
    return lab


def _speech_run(utterances, handle, min_speech_ms, min_silence_ms, pad_ms, feat_mode, sample_rate):
    handle = handle or runtime.default_handle()
    if not handle.has_classifier:
        raise RuntimeError("set FFN weights first (Handle.set_ffn_weights)")
    for v in (min_speech_ms, min_silence_ms, pad_ms):
        runtime.speech_ms_to_rows(v)               # argument errors before any device work
    pcm, offsets, lengths = _upload_16k(utterances, handle, sample_rate)
    plan = runtime.Plan(handle, offsets, lengths, MODE_VAD)
    labels, _, _ = plan.vad(pcm, feat_mode=feat_mode)
    segs, seg_off, sp_off, _ = plan.speech_segments(labels, min_speech_ms, min_silence_ms, pad_ms)
    return plan, pcm, segs, seg_off, sp_off


def source_bounds(segments, n, sample_rate):
    """[start, end) bounds at 16 kHz -> the same speech at ``sample_rate`` in an utterance of ``n`` samples there:
    [floor(a down / up), min(n, ceil(b down / up)))."""
    s = np.asarray(segments, dtype=np.int64).reshape(-1, 2)
    g = int(np.gcd(int(sample_rate), config.SAMPLERATE))
    up, down = config.SAMPLERATE // g, int(sample_rate) // g
    a = s[:, 0] * down // up
    b = np.minimum(int(n), -((-s[:, 1] * down) // up))
    return np.stack([a, b], axis=1)


def speech_segments(utterances, handle=None, min_speech_ms=0, min_silence_ms=0, pad_ms=0, feat_mode=FEAT_ANALYSER,
                    sample_rate=16000):
    """Speech segments of every utterance: a list of int64 [k, 2] arrays of [start, end) samples within the
    utterance.  One upload, the fused VAD, the segment kernels and one download; the handle's front end and
    decision threshold apply.  See Plan.speech_segments for the smoothing parameters.  At any other ``sample_rate``
    the batch is resampled to 16 kHz on the device first and the bounds come back in the caller's rate
    (``source_bounds``)."""
    _, _, segs, seg_off, _ = _speech_run(utterances, handle, min_speech_ms, min_silence_ms, pad_ms, feat_mode,
                                         sample_rate)
    s = segs.cpu().numpy()
    out = [s[seg_off[u]:seg_off[u + 1]] for u in range(len(seg_off) - 1)]
    if int(sample_rate) == config.SAMPLERATE:
        return out
    return [source_bounds(b, len(u), sample_rate) for b, u in zip(out, utterances)]


def extract_speech(utterances, handle=None, min_speech_ms=0, min_silence_ms=0, pad_ms=0, feat_mode=FEAT_ANALYSER,
                   sample_rate=16000):
    """Speech-only audio of every utterance (its segments concatenated): a list of int16 arrays.  The audio is at
    16 kHz whatever ``sample_rate`` the input has: it is the resampled signal the decisions were made on."""
    plan, pcm, segs, seg_off, sp_off = _speech_run(utterances, handle, min_speech_ms, min_silence_ms, pad_ms, feat_mode,
                                                   sample_rate)
    out = plan.gather_speech(pcm, segs, seg_off, sp_off).cpu().numpy()
    return [out[sp_off[u]:sp_off[u + 1]] for u in range(len(sp_off) - 1)]


# ---- drop-ins for dataset/file_processing.py ---------------------------------------------------
def parse_transcription(path, frame_rate):
    """dataset/file_processing.py:106-107 -> dataset/stm_parser.py:5-26."""
    return parse_stm(path, frame_rate)


def _gather_segments(data, transcription_path, frame_rate):
    if transcription_path and frame_rate:
        starts, ends = parse_transcription(transcription_path, frame_rate)
        parts = [data[s:e] for s, e in zip(starts, ends)]
        return np.concatenate(parts).astype(np.int16) if parts else np.array([], dtype=np.int16)
    if transcription_path and frame_rate is None:
        raise Exception('You must specify frame_rate')
    return data


def split_into_frames(data, frame_size, step, transcription_path=None, frame_rate=None):
    """dataset/file_processing.py:80-103: list of overlapping views, strict '>' end rule."""
    data = _gather_segments(np.asarray(data), transcription_path, frame_rate)
    frames = []
    offset = 0
    while len(data) - offset > frame_size:
        frames.append(data[offset:offset + frame_size])
        offset += step
    return frames


class FileFeatures(list):
    """process_file's return value: a list of (mfcc, d1, d2) float64 triples, T-5 long, exactly as the reference
    builds it -- but every triple is a VIEW into one contiguous ``rows`` array [T-5, 39], so ``scale_features`` and
    the sinks can treat a whole file as one array instead of walking 39 x frames python objects."""

    def __init__(self, rows):
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        list.__init__(self, [(r[:13], r[13:26], r[26:]) for r in rows])
        self.rows = rows


def _check_frame_args(frame_size, frame_step, fft_n, mel_filterbank, mfcc_num):
    if int(frame_size) != config.FRAME_SIZE or int(frame_step) != config.FRAME_STEP:
        raise NotImplementedError("vad_b200 kernels are compiled for frame 400 / step 160 (config.py:21-22)")
    from . import mfcc as _mfcc
    _mfcc._require(fft_n, mel_filterbank, mfcc_num)


def _dataset_rows_of_files(jobs, handle, resample=False):
    """[(fname, transcription_path)] -> (device rows [sum, 39], row_offsets): container parse on the host, then one
    upload, ``vadb200_ingest_pcm`` (decode + .stm gather) and one MODE_DATASET launch for the whole step
    (``resample``: DeviceIngest's decode and 16 kHz resampling of other formats and rates)."""
    ing = DeviceIngest(handle, resample=resample)
    for fname, tpath in jobs:
        ing.add(fname, tpath)
    d_pcm, offsets, lengths, _ = ing.run()
    plan = runtime.Plan(handle, offsets, lengths, MODE_DATASET)
    return plan.mfcc(d_pcm), plan.row_offsets


def process_file(args):
    """dataset/file_processing.py:14-77.  args = [fname, frame_size, frame_step, fft_n, mel_filterbank,
    mfcc_num, counter_queue, transcription_path]; returns the list of (mfcc, d1, d2) float64 triples, T-5 long.
    File decode (wav / NIST SPHERE), .stm segment gather, the frame loop, ring and deltas all run on the GPU."""
    fname, frame_size, frame_step, fft_n, mel_filterbank, mfcc_num, counter_queue, transcription_path = args[:8]
    if not (fname.endswith(".wav") or fname.endswith(".sph")):
        raise ValueError("Wrong file format: " + str(fname))
    _check_frame_args(frame_size, frame_step, fft_n, mel_filterbank, mfcc_num)
    rows, _ = _dataset_rows_of_files([(fname, transcription_path)], runtime.default_handle())
    features = FileFeatures(rows.cpu().numpy())
    if counter_queue is not None:
        processed_files = counter_queue.get() + 1
        if processed_files % 5 == 0:
            print("Processed " + str(processed_files) + ' files')
        counter_queue.put(processed_files)
    return features


def scale_features(features, handle=None):
    """dataset/utils.py:5-32: in-place z-score with one scalar mean / population std per group (mfcc, d1, d2) over
    every frame x coefficient of the step.  The reduction (float64 accumulation) and the normalisation run in the
    ``vadb200_scale_rows`` kernels on the packed [n, 39] rows; files produced by ``process_file`` are written back
    with one array assignment each (their triples are views), foreign containers with one assignment per triple."""
    handle = handle or runtime.default_handle()
    blocks = []
    for ff in features:
        if isinstance(ff, FileFeatures):
            blocks.append(ff.rows)
        elif len(ff):
            blocks.append(np.concatenate([np.concatenate(fr) for fr in ff]).reshape(len(ff), -1))
        else:
            blocks.append(np.zeros((0, 39)))
    n = sum(b.shape[0] for b in blocks)
    if n == 0:
        return features
    host = torch.from_numpy(np.concatenate(blocks, axis=0).astype(np.float32))
    dev_rows = host.to(handle.device)
    handle.scale_rows(dev_rows, want_stats=False)
    scaled = dev_rows.cpu().numpy().astype(np.float64)
    pos = 0
    for ff, b in zip(features, blocks):
        part = scaled[pos:pos + b.shape[0]]
        pos += b.shape[0]
        if isinstance(ff, FileFeatures):
            ff.rows[:] = part                      # every (mfcc, d1, d2) view of the file sees it
        else:
            for fr, r in zip(ff, part):
                fr[0][:], fr[1][:], fr[2][:] = r[:13], r[13:26], r[26:]
    return features


# ---- feature sink (file_processing.py:110-148) -----------------------------------------------------------
def create_table_header(mfcc_len):
    """dataset/file_processing.py:110-127: 13 'MFCC Coef', 13 'First delta', 13 'Second delta', 'voiced'."""
    header = ['MFCC Coef' + str(i + 1) for i in range(mfcc_len)]
    header += ['First delta' + str(i + 1) for i in range(mfcc_len)]
    header += ['Second delta' + str(i + 1) for i in range(mfcc_len)]
    header.append('voiced')
    return header


def write_features(writer, features, label):
    """dataset/file_processing.py:130-148: one CSV row per frame, 39 features then the class label."""
    for file_features in features:
        if isinstance(file_features, FileFeatures):
            write_feature_rows(writer, file_features.rows, label)
        else:
            writer.writerows([np.concatenate((ff[0], ff[1], ff[2], [label])) for ff in file_features])


def write_feature_rows(writer, rows, label):
    """Same sink for packed [n, 39] rows (tensor or array)."""
    arr = rows.detach().cpu().numpy() if torch.is_tensor(rows) else np.asarray(rows)
    if arr.shape[0] == 0:
        return
    lab = np.full((arr.shape[0], 1), label, dtype=arr.dtype)
    writer.writerows(np.concatenate([arr, lab], axis=1))


class FeatureStore(object):
    """Binary alternative to the CSV sink: float32 rows [n, 40] = 39 features + class label, appended to
    ``<path>.f32`` with a JSON sidecar ``<path>.json`` (row count, layout).  ``load_feature_store`` memory-maps it
    back (replaces file_processing.load_csv + the h5py line index for the trainer)."""

    WIDTH = 40

    def __init__(self, path, mode="w"):
        self.path = path
        self.rows = 0
        if mode == "a" and os.path.isfile(path + ".json"):
            with open(path + ".json") as f:
                self.rows = int(json.load(f)["rows"])
        self._f = open(path + ".f32", "ab" if mode == "a" else "wb")
        self._flush_meta()

    def _flush_meta(self):
        with open(self.path + ".json", "w") as f:
            json.dump({"rows": self.rows, "width": self.WIDTH, "dtype": "float32",
                       "columns": create_table_header(13)}, f)

    def writerows(self, rows):          # csv.writer duck type: rows of 40 numbers
        arr = np.asarray(rows, dtype=np.float32).reshape(-1, self.WIDTH)
        self._f.write(arr.tobytes())
        self.rows += arr.shape[0]

    def close(self):
        self._f.close()
        self._flush_meta()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def load_feature_store(path):
    with open(path + ".json") as f:
        meta = json.load(f)
    data = np.memmap(path + ".f32", dtype=np.float32, mode="r", shape=(int(meta["rows"]), int(meta["width"])))
    return data[:, :39], data[:, 39].astype(np.int32)


# ---- dataset_creator.process_files (dataset_creator.py:19-73) ------------------------------------------------
def list_audio_files(files_paths, max_files):
    files2process = []
    for files_path in files_paths:
        files2process.extend([files_path + '/' + f for f in os.listdir(files_path)
                              if (f.endswith('.wav') or f.endswith('.sph'))])
    return files2process[:max_files] if len(files2process) > max_files else files2process


def process_files(files_paths, files_type, max_files, csv_writer, transcription_dir=None, handle=None,
                  files_per_step=None, verbose=True, resample=False):
    """dataset_creator.process_files: list wav / sph files of the given directories (os.listdir order, at most
    max_files), derive each file's .stm path from transcription_dir, and for every step of FILES_PER_STEP files
    (config.py:32) extract the (mfcc, d1, d2) rows, scale them with the step's scalar statistics
    (dataset/utils.py:5-32) and write rows + label to ``csv_writer`` (anything with ``writerows``).

    Where the reference maps process_file over a 4-process pool and pickles python lists back, one step here is:
    container headers parsed on the host, one pinned upload of the raw bytes, device decode + .stm gather, one
    MODE_DATASET launch for all files, the two-pass scaling kernels, one download.  The next step's files are read
    from disk while the GPU works on the current one.  Returns the number of rows written.

    ``resample=True`` accepts wav files of any common format, channel count and sample rate and resamples them to
    16 kHz on the device (``DeviceIngest(resample=True)``); the default reads 16 kHz 16-bit mono as the reference
    does."""
    handle = handle or runtime.default_handle()
    step = int(files_per_step or config.FILES_PER_STEP)
    if verbose:
        print("Creating files list...")
    files2process = list_audio_files(files_paths, max_files)
    if verbose:
        print("Need to process %d files" % len(files2process))
    jobs = []
    for file_path in files2process:
        tpath = None
        if transcription_dir is not None:
            tpath = transcription_dir + '/' + file_path.split('/')[-1].split('.')[0] + '.stm'
        jobs.append((file_path, tpath))
    if verbose:
        print("Start processing files...")
    written = 0
    pending = None                                   # (device rows of the previous step), scaled, not yet sunk
    for lo in range(0, len(jobs), step):
        rows, _ = _dataset_rows_of_files(jobs[lo:lo + step], handle, resample)     # enqueued asynchronously
        if rows.shape[0]:
            handle.scale_rows(rows, want_stats=False)
        if pending is not None:                      # sink step k-1 while step k runs on the GPU
            write_feature_rows(csv_writer, pending, files_type)
            written += int(pending.shape[0])
        pending = rows
    if pending is not None:
        write_feature_rows(csv_writer, pending, files_type)
        written += int(pending.shape[0])
    if verbose:
        print("All files are done")
    return written
