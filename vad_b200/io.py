"""Ingest side of the hot path: container parsing on the host (a few header bytes per file), sample decode
and segment gathering on the device.

* ``read_sph`` / ``sph_layout`` restate dataset/sph.py:33-63 (NIST SPHERE).  The reference decodes
  ``sample_count`` big-endian samples starting RIGHT AFTER THE NINTH HEADER LINE -- not at the declared header
  size -- and always most-significant-byte first; ``reference_compat=True`` (default) reproduces exactly that
  byte stream so files give the reference's samples, ``False`` parses the header properly.
* ``wav_layout`` finds the 16-bit mono PCM payload of a RIFF/WAVE file (scipy.io.wavfile.read in
  dataset/file_processing.py:26-27).
* ``wav_format`` reads the layout of any common WAV payload (8/16/24/32-bit PCM, 32/64-bit float, any channel count,
  WAVE_FORMAT_EXTENSIBLE too) for ``DeviceIngest(resample=True)``, which decodes it and resamples it to 16 kHz on the
  device (DESIGN.md section 5.8).
* ``parse_stm`` restates dataset/stm_parser.py:5-26.
* ``DeviceIngest`` stages the raw bytes of many files in ONE pinned buffer, uploads them with one asynchronous
  copy and runs ``vadb200_ingest_pcm`` (byte-swap + STM range gather, dataset/file_processing.py:87-94) into the
  packed, 8-sample-aligned int16 layout the fused kernels read.
"""
import os

import numpy as np
import torch

ALIGN = 8


# ------------------------------------------------------------------------------------------ containers
def sph_layout(fname, reference_compat=True):
    """-> (sample_rate, data_byte_offset, n_samples, big_endian) of a 16-bit NIST SPHERE file."""
    size = os.path.getsize(fname)
    with open(fname, "rb") as f:
        if reference_compat:
            header = [f.readline(1024) for _ in range(9)]                 # dataset/sph.py:36-38
            try:
                samples_num = int(header[2].split(b" ")[2])               # :40
                sample_width = int(header[3].split(b" ")[2])              # :41
                framerate = int(header[6].split(b" ")[2])                 # :43
            except (IndexError, ValueError):
                raise ValueError("not a NIST SPHERE file the reference reader accepts: " + fname)
            if sample_width != 2:
                raise NotImplementedError("only 16-bit SPHERE PCM is supported")
            offset = f.tell()                                             # decoding starts here (:47)
            # samples_num samples, zeros where the file ends early (np.zeros at :45); always MSB first (:55-57)
            return framerate, offset, samples_num, True
        head = f.read(1024)
        if not head.startswith(b"NIST_1A"):
            raise ValueError("not a NIST SPHERE file: " + fname)
        hsize = int(head.split(b"\n")[1].strip())
        if hsize > 1024:
            head += f.read(hsize - 1024)
    fields = {}
    for line in head.split(b"\n")[2:]:
        parts = line.strip().split()
        if not parts or parts[0] == b"end_head":
            break
        if len(parts) >= 3:
            fields[parts[0].decode()] = parts[2].decode()
    if int(fields.get("sample_n_bytes", 2)) != 2:
        raise NotImplementedError("only 16-bit SPHERE PCM is supported")
    n = min(int(fields.get("sample_count", (size - hsize) // 2)), (size - hsize) // 2)
    return int(fields.get("sample_rate", 16000)), hsize, n, fields.get("sample_byte_format", "10") == "10"


def read_sph(fname, reference_compat=True):
    """Host decode (small files, tests): -> (sample_rate, int16[n])."""
    rate, off, n, be = sph_layout(fname, reference_compat)
    avail = max(0, min(2 * n, (os.path.getsize(fname) - off) // 2 * 2))
    raw = np.zeros(2 * n, dtype=np.uint8)
    raw[:avail] = np.fromfile(fname, dtype=np.uint8, count=avail, offset=off)
    return rate, raw.view(">i2" if be else "<i2").astype(np.int16)


def wav_layout(fname):
    """-> (sample_rate, data_byte_offset, n_samples) of a 16-bit mono PCM RIFF/WAVE file."""
    with open(fname, "rb") as f:
        head = f.read(12)
        if len(head) < 12 or head[:4] != b"RIFF" or head[8:12] != b"WAVE":
            raise ValueError("not a RIFF/WAVE file: " + fname)
        fmt = None
        while True:
            ck = f.read(8)
            if len(ck) < 8:
                raise ValueError("no data chunk in " + fname)
            cid, csz = ck[:4], int.from_bytes(ck[4:8], "little")
            if cid == b"fmt ":
                body = f.read(csz + (csz & 1))
                fmt = (int.from_bytes(body[0:2], "little"), int.from_bytes(body[2:4], "little"),
                       int.from_bytes(body[4:8], "little"), int.from_bytes(body[14:16], "little"))
            elif cid == b"data":
                if fmt is None:
                    raise ValueError("data chunk before fmt chunk in " + fname)
                tag, channels, rate, bits = fmt
                if tag not in (1, 0xFFFE) or channels != 1 or bits != 16:
                    raise NotImplementedError("vad_b200 ingests 16-bit mono PCM wav files only: " + fname)
                off = f.tell()
                avail = os.path.getsize(fname) - off
                return rate, off, min(csz, avail) // 2
            else:
                f.seek(csz + (csz & 1), 1)


# (format tag, bits per sample) -> VADB200_PCM_* (runtime.PCM_*)
_WAV_FORMATS = {(1, 8): 1, (1, 16): 0, (1, 24): 2, (1, 32): 3, (3, 32): 4, (3, 64): 5}
_PCM_BYTES = {0: 2, 1: 1, 2: 3, 3: 4, 4: 4, 5: 8}


def wav_format(fname):
    """-> (sample_rate, data_byte_offset, n_frames, channels, fmt) of a RIFF/WAVE file holding integer PCM (tag 1: 8-bit
    unsigned, 16 / 24 / 32-bit signed), IEEE float (tag 3: 32 / 64 bit) or WAVE_FORMAT_EXTENSIBLE with either
    subformat; ``fmt`` is a VADB200_PCM_* code (runtime.PCM_*).  Frames past the end of a truncated file are not
    counted."""
    with open(fname, "rb") as f:
        head = f.read(12)
        if len(head) < 12 or head[:4] != b"RIFF" or head[8:12] != b"WAVE":
            raise ValueError("not a RIFF/WAVE file: " + fname)
        fmt = None
        while True:
            ck = f.read(8)
            if len(ck) < 8:
                raise ValueError("no data chunk in " + fname)
            cid, csz = ck[:4], int.from_bytes(ck[4:8], "little")
            if cid == b"fmt ":
                body = f.read(csz + (csz & 1))
                if len(body) < 16:
                    raise ValueError("short fmt chunk in " + fname)
                tag = int.from_bytes(body[0:2], "little")
                if tag == 0xFFFE:
                    if len(body) < 40:
                        raise ValueError("short WAVE_FORMAT_EXTENSIBLE fmt chunk in " + fname)
                    tag = int.from_bytes(body[24:26], "little")       # first two bytes of the subformat GUID
                fmt = (tag, int.from_bytes(body[2:4], "little"), int.from_bytes(body[4:8], "little"),
                       int.from_bytes(body[14:16], "little"))
            elif cid == b"data":
                if fmt is None:
                    raise ValueError("data chunk before fmt chunk in " + fname)
                tag, channels, rate, bits = fmt
                code = _WAV_FORMATS.get((tag, bits))
                if code is None or not 1 <= channels <= 32:
                    raise NotImplementedError("unsupported wav format (tag %d, %d bits, %d channels): %s"
                                              % (tag, bits, channels, fname))
                off = f.tell()
                avail = os.path.getsize(fname) - off
                return rate, off, min(csz, avail) // (_PCM_BYTES[code] * channels), channels, code
            else:
                f.seek(csz + (csz & 1), 1)


def parse_stm(path, frame_rate):
    """dataset/stm_parser.py:5-26: TED-LIUM .stm segment bounds in samples.  Lines with fewer than 7 fields or
    labelled ignore_time_segment_in_scoring are skipped; seconds are float32 and the product is truncated to int32."""
    starts, ends = [], []
    with open(path, "r") as f:
        for line in f:
            items = line.split(" ")
            if len(items) < 7 or items[6].strip() == "ignore_time_segment_in_scoring":
                continue
            starts.append(np.float32(items[3]))
            ends.append(np.float32(items[4]))
    s = (np.array(starts, dtype=np.float32) * frame_rate).astype(np.int32)
    e = (np.array(ends, dtype=np.float32) * frame_rate).astype(np.int32)
    return s, e


def clip_ranges(starts, ends, n):
    """numpy slice semantics of ``data[start:end]`` (file_processing.py:91-92) for non-negative bounds."""
    s = np.clip(np.asarray(starts, dtype=np.int64), 0, n)
    e = np.clip(np.asarray(ends, dtype=np.int64), 0, n)
    return s, np.maximum(e, s)


# ------------------------------------------------------------------------------------------ device ingest
class DeviceIngest(object):
    """Raw files -> packed int16 PCM on the device.  ``add(path, transcription_path)`` registers a file;
    ``run()`` returns (d_pcm int16 tensor, offsets, lengths, sample_rates).

    ``resample=True`` also takes wav files of any format ``wav_format`` reads and any supported sample rate: each file
    is decoded on the device (``vadb200_decode_pcm``: float32 in int16 units, the mean of its channels), its .stm
    segments are gathered at its own rate, and the concatenation is resampled to 16 kHz (``runtime.Resampler``).
    ``run()`` then returns 16 kHz offsets and lengths, and 16000 as every file's rate.  A 16 kHz mono 16-bit file
    takes the ``vadb200_ingest_pcm`` path as without resampling, so its samples are the same."""

    def __init__(self, handle, resample=False):
        self.handle = handle
        self.resample = bool(resample)
        # (path, byte_offset, n_frames, big_endian, seg_starts, seg_ends, rate, channels, fmt)
        self.files = []

    def add(self, fname, transcription_path=None):
        channels, fmt = 1, 0
        if fname.endswith(".wav"):
            if self.resample:
                rate, off, n, channels, fmt = wav_format(fname)
            else:
                rate, off, n = wav_layout(fname)
            be = False
        elif fname.endswith(".sph"):
            rate, off, n, be = sph_layout(fname)
        else:
            raise ValueError("Wrong file format: " + str(fname))
        if self.resample:
            from .runtime import resampled_length
            resampled_length(0, rate)                       # an unsupported rate fails here, before any upload
        if transcription_path:
            s, e = parse_stm(transcription_path, rate)
            if np.any(s < 0) or np.any(e < 0):
                raise NotImplementedError("negative .stm bounds (python negative slicing) are not supported")
            s, e = clip_ranges(s, e, n)
        else:
            s, e = np.array([0], dtype=np.int64), np.array([n], dtype=np.int64)
        self.files.append((fname, off, n, be, s, e, rate, channels, fmt))

    def run(self):
        if self.resample:
            return self._run_resample()
        h = self.handle
        raw_off, pos = [], 0
        for (_, _, n, _, _, _, _, _, _) in self.files:    # 2-byte aligned slot per file in the raw stream
            raw_off.append(pos)
            pos += 2 * n + (2 * n) % 4
        raw = torch.zeros(max(pos, 4), dtype=torch.uint8).pin_memory()   # zeros: a short file leaves a silent tail
        rawv = raw.numpy()
        lengths = np.zeros(len(self.files), dtype=np.int64)
        seg_src, seg_dst, seg_len, seg_be = [], [], [], []
        for i, (fname, off, n, be, s, e, _, _, _) in enumerate(self.files):
            with open(fname, "rb") as f:
                f.seek(off)
                f.readinto(memoryview(rawv[raw_off[i]:raw_off[i] + 2 * n]))   # reads what the file has
            lengths[i] = int((e - s).sum())
        padded = (lengths + ALIGN - 1) // ALIGN * ALIGN
        offsets = np.zeros(len(self.files), dtype=np.int64)
        if len(self.files) > 1:
            offsets[1:] = np.cumsum(padded[:-1])
        for i, (_, _, _, be, s, e, _, _, _) in enumerate(self.files):
            d = offsets[i]
            for a, b in zip(s, e):
                if b > a:
                    seg_src.append(raw_off[i] // 2 + int(a))
                    seg_dst.append(int(d))
                    seg_len.append(int(b - a))
                    seg_be.append(be)
                    d += int(b - a)
        total = int(padded.sum()) + ALIGN
        d_raw = raw.to(h.device, non_blocking=True)
        d_pcm = torch.zeros(total, dtype=torch.int16, device=h.device)
        seg_src, seg_dst, seg_len = (np.asarray(x, dtype=np.int64) for x in (seg_src, seg_dst, seg_len))
        seg_be = np.asarray(seg_be, dtype=bool)
        for be in (False, True):
            m = seg_be == be
            for lo in range(0, int(m.sum()), 65535):
                sl = slice(lo, lo + 65535)
                h.ingest_pcm(d_raw, seg_src[m][sl], seg_dst[m][sl], seg_len[m][sl], d_pcm, big_endian=be)
        rates = [f[6] for f in self.files]
        return d_pcm, offsets, lengths, rates

    def _run_resample(self):
        from .runtime import Resampler, resampled_length
        h = self.handle
        direct = [f[6] == 16000 and f[7] == 1 and f[8] == 0 for f in self.files]   # 16 kHz mono s16: ingest_pcm
        raw_off, pos = [], 0
        for (_, _, n, _, _, _, _, ch, fmt) in self.files:   # slots aligned to 8 bytes and to the file's frame size
            fb = _PCM_BYTES[fmt] * ch
            unit = 8 * fb // np.gcd(8, fb)
            pos = (pos + unit - 1) // unit * unit
            raw_off.append(pos)
            pos += n * fb
        raw = torch.zeros(max(pos, 8), dtype=torch.uint8).pin_memory()
        rawv = raw.numpy()
        src_len = np.zeros(len(self.files), dtype=np.int64)
        for i, (fname, off, n, _, s, e, _, ch, fmt) in enumerate(self.files):
            with open(fname, "rb") as f:
                f.seek(off)
                f.readinto(memoryview(rawv[raw_off[i]:raw_off[i] + n * _PCM_BYTES[fmt] * ch]))
            src_len[i] = int((e - s).sum())
        lengths = np.array([l if d else resampled_length(l, f[6]) for l, d, f in zip(src_len, direct, self.files)],
                           dtype=np.int64)
        padded = (lengths + ALIGN - 1) // ALIGN * ALIGN
        offsets = np.zeros(len(self.files), dtype=np.int64)
        if len(self.files) > 1:
            offsets[1:] = np.cumsum(padded[:-1])
        f_off = np.zeros(len(self.files), dtype=np.int64)      # decoded float32 staging at the source rate
        if len(self.files) > 1:
            f_off[1:] = np.cumsum(np.where(direct, 0, src_len)[:-1])
        d_raw = raw.to(h.device, non_blocking=True)
        d_pcm = torch.zeros(int(padded.sum()) + ALIGN, dtype=torch.int16, device=h.device)
        d_f32 = torch.empty(max(int(np.where(direct, 0, src_len).sum()), 1), dtype=torch.float32, device=h.device)
        groups = {}                                             # (direct, fmt, channels, big_endian) -> segments
        for i, (_, _, _, be, s, e, _, ch, fmt) in enumerate(self.files):
            fb = _PCM_BYTES[fmt] * ch
            d = int(offsets[i]) if direct[i] else int(f_off[i])
            g = groups.setdefault((direct[i], fmt, ch, bool(be)), ([], [], []))
            for a, b in zip(s, e):
                if b > a:
                    g[0].append((raw_off[i] // 2 if direct[i] else raw_off[i] // fb) + int(a))
                    g[1].append(d)
                    g[2].append(int(b - a))
                    d += int(b - a)
        for (is_direct, fmt, ch, be), (src, dst, ln) in groups.items():
            for lo in range(0, len(ln), 65535):
                sl = slice(lo, lo + 65535)
                if is_direct:
                    h.ingest_pcm(d_raw, src[sl], dst[sl], ln[sl], d_pcm, big_endian=be)
                else:
                    h.decode_pcm(d_raw, fmt, ch, src[sl], dst[sl], ln[sl], d_f32, big_endian=be)
        resamplers = {}
        for i, f in enumerate(self.files):
            if direct[i] or src_len[i] == 0:
                continue
            r = resamplers.get(f[6]) or resamplers.setdefault(f[6], Resampler(h, f[6]))
            o = int(offsets[i])
            r.run(d_f32, [int(f_off[i])], [int(src_len[i])], out=d_pcm[o:o + int(padded[i])])
        return d_pcm, offsets, lengths, [16000] * len(self.files)
