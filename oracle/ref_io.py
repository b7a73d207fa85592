"""CPU restatement of the reference's ingest and offline driver (TEST INFRASTRUCTURE).

Line citations are relative to /root/reference.  ``dataset/sph.py`` and ``dataset/stm_parser.py`` are python-2
byte-string code (``header[2].split(' ')`` on a file opened 'rb', ``ord(chunk[i])``) and do not run under
python 3 even through the shim, so these two are restated from the source and are NOT pinned to an execution of
the reference ("parity unpinned" for SPHERE / STM ingest); ``process_file`` on wav files IS pinned to the
reference's own output (tests/golden/utterances.npz) in tests/test_oracle.py.
"""
import os

import numpy as np

from . import ref_math as rm


def read_sph(fname):
    """dataset/sph.py:33-63, byte for byte: nine ``readline(1024)`` header lines, fields taken from lines 2, 3, 4, 6
    (third space-separated token), then ``samples_num`` samples decoded MOST-significant byte first starting at the
    current file position -- i.e. right after the ninth header line, not at the declared header size."""
    with open(fname, "rb") as f:
        header = [f.readline(1024) for _ in range(9)]                      # :36-38
        samples_num = int(header[2].split(b" ")[2])                        # :40
        sample_width = int(header[3].split(b" ")[2])                       # :41
        channels = int(header[4].split(b" ")[2])                           # :42
        framerate = int(header[6].split(b" ")[2])                          # :43
        samples = np.zeros((samples_num,), dtype=np.int16)                 # :45
        counter = 0
        while counter < samples_num:                                       # :48-61 (chunked there)
            chunk = f.read(1024 * sample_width)
            if not chunk:
                break
            if counter + len(chunk) > samples_num:                         # :49-50 (sic: samples vs bytes)
                chunk = chunk[:(samples_num - counter) * sample_width]
            for i in range(len(chunk) // sample_width):                    # :52-58
                sample = 0
                for j in range(sample_width):
                    sample |= chunk[i * sample_width + j] << 8 * (sample_width - 1 - j)
                samples[counter] = np.array(sample, dtype=np.uint16).astype(np.int16) if sample_width == 2 else sample
                counter += 1
    return channels, framerate, sample_width, samples


def stm_sample_indices(fname, samplerate):
    """dataset/stm_parser.py:5-26."""
    starts = np.array([], dtype=np.float32)
    ends = np.array([], dtype=np.float32)
    with open(fname, "r") as f:
        for chunk in f:
            items = chunk.split(" ")
            if (len(items) < 7) or (items[6].strip() == "ignore_time_segment_in_scoring"):
                continue
            starts = np.append(starts, np.float32(items[3]))
            ends = np.append(ends, np.float32(items[4]))
    return (starts * samplerate).astype(np.int32), (ends * samplerate).astype(np.int32)


def file_samples(fname, transcription_path=None):
    """What ``process_file`` frames (dataset/file_processing.py:26-38, 87-94): decoded samples, .stm segments glued."""
    if fname.endswith(".wav"):
        from scipy.io import wavfile
        rate, data = wavfile.read(fname)
    elif fname.endswith(".sph"):
        _, rate, _, data = read_sph(fname)
    else:
        raise ValueError("Wrong file format: " + str(fname))
    if transcription_path:
        starts, ends = stm_sample_indices(transcription_path, rate)
        new_data = np.array([], dtype=np.int16)
        for s, e in zip(starts, ends):
            new_data = np.append(new_data, data[s:e])
        data = new_data
    return np.asarray(data, dtype=np.int16)


def process_files_rows(files_paths, max_files, transcription_dir=None, files_per_step=30):
    """dataset_creator.py:19-73 as arrays: for every step of ``files_per_step`` files the scaled [n, 39] rows
    (dataset/utils.py:5-32), concatenated in file order."""
    files = []
    for d in files_paths:
        files.extend([d + '/' + f for f in os.listdir(d) if (f.endswith('.wav') or f.endswith('.sph'))])
    files = files[:max_files] if len(files) > max_files else files
    out = []
    for lo in range(0, len(files), files_per_step):
        groups = []
        for fp in files[lo:lo + files_per_step]:
            tp = None
            if transcription_dir is not None:
                tp = transcription_dir + '/' + fp.split('/')[-1].split('.')[0] + '.stm'
            groups.append(rm.dataset_features(rm.mfcc_utterance(file_samples(fp, tp))))
        if sum(g.shape[0] for g in groups):
            scaled, _ = rm.scale_features(groups)
            out.extend(scaled)
    return np.concatenate(out, axis=0) if out else np.zeros((0, 39)), files
