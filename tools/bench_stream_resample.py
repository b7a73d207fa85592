"""Tick cost of the resampling ragged bank: 4096 streams through the captured-graph, zero-copy tick, host wall clock
per tick (one graph launch + synchronise), as tools/bench_stream_ragged.py times the 16 kHz ragged bank.  Workloads,
alternated round by round in one process:

  16k_160        the 16 kHz ragged bank, 160 samples a stream (cap 160): the baseline
  8k_80 / 8k_160 8 kHz (telephony), 10 / 20 ms packets (cap = the packet)
  44k1_441       44.1 kHz, 10 ms packets
  48k_480 / 48k_960   48 kHz (WebRTC, sound cards), 10 / 20 ms packets
  48k_jitter     48 kHz, each stream draws 0, 480 or 960 samples a tick (mean 10 ms; cap 960)

The packets of each tick are packed into the bank's pinned buffers before the clock starts.  Per workload: p50 / p99 /
max tick in ms, the PCIe bytes of packets a tick reads, and rows per second (rows emitted over the summed tick
time).  After the timed rounds, a separate torch.profiler pass over 200 ticks per workload gives the
device time of the resampling steps alone (stream_resample_plan_kernel + stream_resample_kernel) and of the unchanged
stream_ragged_kernel after them, per tick.  Prints one JSON object with the card's name, power limit and max SM clock
read in the same process, and writes it to --out when given.

    python tools/bench_stream_resample.py --ticks 3000 --out profiles/r10_stream_resample_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_math as rm  # noqa: E402
from vad_b200 import runtime  # noqa: E402
from vad_b200.analyser import StreamBank  # noqa: E402

N = 4096
POOL = 16      # distinct ticks per workload, cycled
# name -> (rate, cap, packet sizes drawn per stream)
WORKLOADS = {
    "16k_160": (16000, 160, [160]),
    "8k_80": (8000, 80, [80]),
    "8k_160": (8000, 160, [160]),
    "44k1_441": (44100, 441, [441]),
    "48k_480": (48000, 480, [480]),
    "48k_960": (48000, 960, [960]),
    "48k_jitter": (48000, 960, [0, 480, 960]),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--profile-ticks", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    h = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    rng = np.random.default_rng(0)
    names = list(WORKLOADS)
    banks, ticks = {}, {}
    for name in names:
        rate, cap, sizes = WORKLOADS[name]
        banks[name] = StreamBank(N, handle=h, max_feed_samples=cap, sample_rate=rate)
        pool = []
        for _ in range(POOL):
            s = rng.choice(sizes, size=N)
            off = np.r_[0, np.cumsum(s)].astype(np.int64)
            pool.append(((rng.standard_normal(int(off[-1])) * 3000).astype(np.int16), off))
        ticks[name] = pool

    def tick(name, t):
        b = banks[name]
        flat, off = ticks[name][t % POOL]
        b.h_samples.numpy()[:flat.size] = flat
        b.h_offsets.numpy()[:] = off
        t0 = time.perf_counter()
        b._tick(False)
        dt = time.perf_counter() - t0
        return dt, flat.size, int(b.h_counts.numpy().clip(0).sum())

    for name in names:                                   # warm-up: captures every graph, fills every state
        for t in range(a.warmup):
            tick(name, t)
    lat = {name: [] for name in names}
    fed = {name: 0 for name in names}
    rows = {name: 0 for name in names}
    per_round = a.ticks // a.rounds
    for r in range(a.rounds):
        for name in names:
            for t in range(per_round):
                dt, k, c = tick(name, r * per_round + t)
                lat[name].append(dt)
                fed[name] += k
                rows[name] += c
    # device time per kernel, in a pass of its own (the profiler slows the host)
    dev = {}
    from torch.profiler import ProfilerActivity, profile
    for name in names:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for t in range(a.profile_ticks):
                tick(name, t)
        us = {"resample_steps": 0.0, "ragged": 0.0}
        for ev in prof.key_averages():       # kernels: their device time is their own
            t = getattr(ev, "device_time_total", None)
            t = ev.cuda_time_total if t is None else t
            if "stream_resample_plan_kernel" in ev.key or "stream_resample_kernel" in ev.key:
                us["resample_steps"] += t
            elif "stream_ragged_kernel" in ev.key:
                us["ragged"] += t
        dev[name] = {k: round(v / a.profile_ticks, 2) for k, v in us.items()}
    res = {"card": card(), "streams": N, "timed_ticks": per_round * a.rounds, "workloads": {}}
    for name in names:
        rate, cap, _ = WORKLOADS[name]
        ms = np.sort(np.asarray(lat[name])) * 1e3
        res["workloads"][name] = {
            "rate": rate, "cap": cap,
            "mean_samples_per_stream": round(fed[name] / (N * len(ms)), 2),
            "pcie_bytes_per_tick": int(2 * fed[name] / len(ms)),
            "p50_ms": round(float(ms[len(ms) // 2]), 4),
            "p99_ms": round(float(ms[int(len(ms) * 0.99)]), 4),
            "max_ms": round(float(ms[-1]), 4),
            "rows_per_s": round(rows[name] / float(ms.sum() / 1e3), 0),
            "resample_steps_us_per_tick": dev[name]["resample_steps"],
            "ragged_kernel_us_per_tick": dev[name]["ragged"],
        }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
