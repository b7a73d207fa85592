"""Tick cost of the ragged stream bank: 4096 streams through the captured-graph, zero-copy tick, host wall clock per
tick (one graph launch + synchronise) as bench.py's stream record times the fixed bank.  Workloads, alternated round
by round in one process:

  fixed_160      the fixed bank, 160 samples a stream (the reference the ragged path is measured against)
  ragged_160     the ragged bank (cap 160), 160 samples a stream
  ragged_320 / _400 / _480   uniform packets of that size (cap = the packet)
  jitter         each stream draws 0, 160 or 320 samples a tick (mean 160; cap 320)
  skew           1 stream in 32 takes 1600 samples, the rest 160 (cap 1600): one busy stream per CTA

The packets of each tick are packed into the bank's pinned buffers before the clock starts.  Per workload: p50 / p99 /
max tick in ms and frames per second (samples fed / 160 over the summed tick time).  Prints one JSON object with the
card's name and power limit read in the same process, and writes it to --out when given.

    python tools/bench_stream_ragged.py --ticks 3000 --out profiles/r8_stream_ragged_bench.json
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def sizes_of(name, rng):
    if name == "jitter":
        return rng.choice([0, 160, 320], size=N)
    if name == "skew":
        s = np.full(N, 160)
        s[rng.permutation(N // 32) * 32 + rng.integers(0, 32, N // 32)] = 1600   # one stream in each CTA
        return s
    return np.full(N, int(name.split("_")[1]))


CAP = {"ragged_160": 160, "ragged_320": 320, "ragged_400": 400, "ragged_480": 480, "jitter": 320, "skew": 1600}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    h = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    rng = np.random.default_rng(0)
    names = ["fixed_160"] + list(CAP)
    banks, ticks = {}, {}
    for name in names:
        if name == "fixed_160":
            banks[name] = StreamBank(N, handle=h)
            ticks[name] = [(rng.standard_normal((N, 160)) * 3000).astype(np.int16) for _ in range(POOL)]
            continue
        b = StreamBank(N, handle=h, max_feed_samples=CAP[name])
        banks[name] = b
        pool = []
        for _ in range(POOL):
            s = sizes_of(name, rng)
            off = np.r_[0, np.cumsum(s)].astype(np.int64)
            pool.append(((rng.standard_normal(int(off[-1])) * 3000).astype(np.int16), off))
        ticks[name] = pool

    def tick(name, t):
        b, x = banks[name], ticks[name][t % POOL]
        if name == "fixed_160":
            b.h_chunks.numpy()[:] = x
            fed = x.size
        else:
            flat, off = x
            b.h_samples.numpy()[:flat.size] = flat
            b.h_offsets.numpy()[:] = off
            fed = flat.size
        t0 = time.perf_counter()
        b._tick(False)
        return time.perf_counter() - t0, fed

    for name in names:                                   # warm-up: captures every graph, fills every ring
        for t in range(a.warmup):
            tick(name, t)
    lat = {name: [] for name in names}
    fed = {name: 0 for name in names}
    per_round = a.ticks // a.rounds
    for r in range(a.rounds):
        for name in names:
            for t in range(per_round):
                dt, k = tick(name, r * per_round + t)
                lat[name].append(dt)
                fed[name] += k
    res = {"card": card(), "streams": N, "timed_ticks": per_round * a.rounds, "workloads": {}}
    for name in names:
        ms = np.sort(np.asarray(lat[name])) * 1e3
        res["workloads"][name] = {
            "cap": CAP.get(name, 160),
            "mean_samples_per_stream": round(fed[name] / (N * len(ms)), 2),
            "p50_ms": round(float(ms[len(ms) // 2]), 4),
            "p99_ms": round(float(ms[int(len(ms) * 0.99)]), 4),
            "max_ms": round(float(ms[-1]), 4),
            "frames_per_s": round(fed[name] / 160 / float(ms.sum() / 1e3), 0),
        }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
