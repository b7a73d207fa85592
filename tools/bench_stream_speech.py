"""Tick cost of speech segments on the stream bank: 4096 streams, speech off vs on at 25/10/3 rows and at
1000/1000/1000 rows (D = 2998), alternated in the same process.  Per configuration: p50 / p99 of the host-timed
feed_pinned tick (one graph launch + synchronise) and of the feed_speech tick (the same plus rows and bounds),
kernel-only device time from CUDA events, and the time to end all 4096 streams at D = 2998.  Prints one JSON object
and writes it to --out when given.

    python tools/bench_stream_speech.py --ticks 3000 --out profiles/r6_stream_speech_bench.json
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
CONFIGS = [("off", None), ("25/10/3", (25, 10, 3)), ("1000/1000/1000", (1000, 1000, 1000))]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def pct(lat):
    ms = np.sort(np.asarray(lat)) * 1e3
    return {"p50_ms": round(float(ms[len(ms) // 2]), 4), "p99_ms": round(float(ms[int(len(ms) * 0.99)]), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=300)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    h = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    banks = {}
    for name, p in CONFIGS:
        b = StreamBank(N, handle=h)
        if p is not None:
            b.set_speech(*(10 * v for v in p))        # rows -> ms
        banks[name] = b
    rng = np.random.default_rng(0)
    pool = torch.from_numpy((rng.standard_normal((32, N, 160)) * 3000).astype(np.int16))
    lat = {(name, k): [] for name, _ in CONFIGS for k in ("feed_pinned", "feed_speech")}
    per_round = a.ticks // a.rounds

    def tick(b, t, speech):
        b.h_chunks.copy_(pool[t % 32])
        t0 = time.perf_counter()
        b._tick(False, speech=speech)
        return time.perf_counter() - t0

    for name, p in CONFIGS:                               # warm-up: captures every graph
        for t in range(a.warmup):
            tick(banks[name], t, False)
            if p is not None:
                tick(banks[name], t, True)
    t_glob = 0
    for _ in range(a.rounds):                             # alternate the configurations
        for name, p in CONFIGS:
            for t in range(per_round):
                lat[(name, "feed_pinned")].append(tick(banks[name], t_glob + t, False))
                if p is not None:
                    lat[(name, "feed_speech")].append(tick(banks[name], t_glob + t, True))
        t_glob += per_round
    res = {"card": card(), "streams": N, "timed_ticks": per_round * a.rounds, "configs": {}}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 500
    for _ in range(2):                                    # kernel-only, alternated twice; the second pass is kept
        for name, p in CONFIGS:
            b = banks[name]
            b.d_chunks.copy_(pool[0].to(b.d_chunks.device))
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(reps):
                if p is None:
                    b.bank.feed_ptr(b.d_chunks.data_ptr(), b.d_labels.data_ptr(), 0)
                else:
                    b.bank.feed_speech_ptr(b.d_chunks.data_ptr(), b.d_labels.data_ptr(), 0, b.d_rows.data_ptr(),
                                           b.d_bounds.data_ptr())
            ev1.record()
            torch.cuda.synchronize()
            res["configs"].setdefault(name, {})["kernel_us"] = round(ev0.elapsed_time(ev1) / reps * 1e3, 3)
    for name, p in CONFIGS:
        c = res["configs"][name]
        c["delay_rows"] = banks[name].delay
        c["feed_pinned"] = pct(lat[(name, "feed_pinned")])
        if p is not None:
            c["feed_speech"] = pct(lat[(name, "feed_speech")])
    # ending every stream at the largest delay: each stream has fed more than D rows, so each drains D rows
    b = banks["1000/1000/1000"]
    D = b.delay
    end = torch.ones((N,), dtype=torch.uint8, device=h.device)
    ends = []
    for i in range(5):
        for t in range(D + 100):                          # refill: every stream holds D pending rows again
            b.bank.feed_ptr(b.d_chunks.data_ptr(), b.d_labels.data_ptr(), 0)
        torch.cuda.synchronize()
        ev0.record()
        b.bank.end_streams_ptr(end.data_ptr(), b.d_tail_rows.data_ptr(), b.d_tail_bounds.data_ptr())
        ev1.record()
        torch.cuda.synchronize()
        ends.append(ev0.elapsed_time(ev1) * 1e3)
        assert int((b.d_tail_rows != 255).sum()) == N * D
    res["end_all_streams"] = {"delay_rows": D, "median_us": round(float(np.median(ends)), 1),
                              "all_us": [round(x, 1) for x in ends]}
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
