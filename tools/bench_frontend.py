#!/usr/bin/env python
"""Cost of the opt-in front end (pre-emphasis 0.97 + Hamming window, and for VAD the threshold 0.5 on p(voiced)):
the default kernels against the front-end variant, alternated in one process, on device-resident synthetic PCM of
several GB (well beyond the 126 MB L2, so every pass reads PCM from HBM).  CUDA events around each launch.
    python tools/bench_frontend.py [--utts 20000] [--reps 7] [--out profiles/r4_frontend_bench.json]
Prints one JSON object (and writes it to --out when given)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_provenance():
    """Card name and power limit by a read-only query."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        out = "nvidia-smi unavailable: %s" % e
    return out


def time_launch(torch, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def ab(torch, h, fn, reps, audio_s, theta):
    """Alternate default / front end; returns per-arm best and median audio-s/s."""
    arms = {"default": [], "frontend": []}
    for arm in ("default", "frontend"):  # warm-up of both variants
        set_arm(h, arm, theta)
        fn()
    torch.cuda.synchronize()
    for _ in range(reps):
        for arm in ("default", "frontend"):
            set_arm(h, arm, theta)
            arms[arm].append(time_launch(torch, fn))
    res = {}
    for arm, ms in arms.items():
        ms = np.array(ms)
        res[arm] = {"ms": [round(float(x), 3) for x in ms], "best_audio_s_per_s": audio_s / (ms.min() * 1e-3),
                    "median_audio_s_per_s": audio_s / (np.median(ms) * 1e-3)}
    res["ratio_best"] = res["frontend"]["best_audio_s_per_s"] / res["default"]["best_audio_s_per_s"]
    res["ratio_median"] = res["frontend"]["median_audio_s_per_s"] / res["default"]["median_audio_s_per_s"]
    return res


def set_arm(h, arm, theta):
    if arm == "default":
        h.set_frontend(0.0, None)
        h.set_decision_threshold(None)
    else:
        h.set_frontend(0.97, "hamming")
        h.set_decision_threshold(theta)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=20000, help="10 s utterances (cfg3 shape); 20000 = 6.4 GB of PCM")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--ticks", type=int, default=2000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_frontend.py measures on the GPU; no CUDA device found")
    from oracle import ref_math as rm
    from vad_b200 import batch, runtime
    from vad_b200.analyser import StreamBank
    h = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    L = 160000
    res = {"gpu": gpu_provenance(), "torch_device": torch.cuda.get_device_name(0), "utterances": a.utts,
           "utt_seconds": 10.0, "reps": a.reps, "frontend": "preemph 0.97, np.hamming(400), threshold 0.5 (VAD)"}
    off, ln, stride = batch.uniform_layout(a.utts, L)
    pcm = h.synth_pcm(a.utts, L, seed=1234, first_utt=0, utt_stride=stride)
    res["pcm_gb"] = pcm.numel() * 2 / 1e9
    audio_s = a.utts * 10.0
    vplan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
    labels = torch.empty((vplan.total_rows,), dtype=torch.uint8, device=h.device)
    res["vad_cfg3"] = ab(torch, h, lambda: vplan.vad(pcm, labels=labels), a.reps, audio_s, 0.5)
    mplan = runtime.Plan(h, off, ln, runtime.MODE_MFCC)
    rows = torch.empty((mplan.total_rows, 13), dtype=torch.float32, device=h.device)
    res["mfcc_cfg2"] = ab(torch, h, lambda: mplan.mfcc(pcm, out=rows), a.reps, audio_s, None)
    del pcm, labels, rows
    # streaming: per-tick latency (graph replay + pinned I/O) at a.streams streams, front end off / on
    rng = np.random.default_rng(0)
    chunks = rng.integers(-3000, 3000, size=(a.streams, 160)).astype(np.int16)
    res["stream"] = {"streams": a.streams, "ticks": a.ticks}
    for arm in ("default", "frontend"):
        set_arm(h, arm, 0.5)
        bank = StreamBank(a.streams, handle=h)        # the tick graph captures the handle's settings
        bank.h_chunks.copy_(torch.from_numpy(chunks))
        for _ in range(50):
            bank.feed_pinned()
        ts = []
        for _ in range(a.ticks):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            bank.feed_pinned()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts = np.array(ts) * 1e3
        res["stream"][arm] = {"p50_us": float(np.percentile(ts, 50)), "p99_us": float(np.percentile(ts, 99))}
        bank.bank.close()
    set_arm(h, "default", None)
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
