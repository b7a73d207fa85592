"""Decision-tree classifier against the FFN on one GPU, in one process (same-box comparison).

  fused VAD   ms per 1000 h of audio and audio-s/s over a device-resident synthetic batch far beyond L2, alternating
              FFN impl 2 (fp16 tcgen05), FFN impl 0 (FP32 cores), the reference-hyperparameter tree and a deep tree;
  tree_predict rows/s at 1 M rows;
  banks       4096-stream fixed and ragged (480-sample packets) ticks, p50 / p99, FFN against the reference tree.

Trees are fitted with sklearn on the device's own features of a slice of the batch (reference grid-search
hyperparameters max_depth=25, min_samples_leaf=20, min_samples_split=22 on the FFN's labels; the deep tree on noisy
labels).  Prints one JSON record (and writes it to --out when given)."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from sklearn.tree import DecisionTreeClassifier  # noqa: E402

from vad_b200 import runtime  # noqa: E402
from vad_b200.analyser import StreamBank  # noqa: E402


def gpu_info():
    import subprocess
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hours", type=float, default=4.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON record to this path")
    a = ap.parse_args()
    torch.cuda.init()
    w = runtime.glorot_ffn(0)
    h = runtime.Handle(0, ffn_weights=w)
    utt = 10 * 16000
    n_utt = int(a.hours * 3600 / 10)
    pcm = h.synth_pcm(n_utt, utt)
    offs = np.arange(n_utt, dtype=np.int64) * utt
    lens = np.full(n_utt, utt, np.int64)
    plan = runtime.Plan(h, offs, lens, runtime.MODE_VAD)
    labels = torch.empty((plan.total_rows,), dtype=torch.uint8, device="cuda")
    # trees, fitted on the device features of the first 200 utterances
    sp = runtime.Plan(h, offs[:200], lens[:200], runtime.MODE_VAD)
    lab, _, ft = sp.vad(pcm, want_feats=True)
    X, y = ft.cpu().numpy(), lab.cpu().numpy()
    ok = np.isfinite(X).all(axis=1)
    X, y = X[ok], y[ok]
    rng = np.random.default_rng(0)
    ref = DecisionTreeClassifier(max_depth=25, min_samples_leaf=20, min_samples_split=22, random_state=0).fit(X, y)
    deep = DecisionTreeClassifier(random_state=0).fit(X, np.where(rng.random(len(y)) < 0.2, 1 - y, y))
    configs = {"ffn_impl2": ("ffn", 2), "ffn_impl0": ("ffn", 0), "tree_ref": ("tree", ref), "tree_deep": ("tree", deep)}

    def setup(kind, arg):
        if kind == "ffn":
            h.clear_tree()
            h.set_ffn_impl(arg)
        else:
            h.set_tree(arg)

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {k: [] for k in configs}
    for rep in range(a.reps + 1):
        for k, (kind, arg) in configs.items():
            setup(kind, arg)
            torch.cuda.synchronize()
            e0.record()
            plan.vad(pcm, labels=labels)
            e1.record()
            torch.cuda.synchronize()
            if rep:
                times[k].append(e0.elapsed_time(e1))
    audio_s = n_utt * 10.0
    fused = {k: dict(ms_median=float(np.median(v)), ms_min=float(np.min(v)),
                     ms_per_1000h=float(np.median(v)) * 1000 * 3600 / audio_s,
                     audio_s_per_s=audio_s / (float(np.median(v)) * 1e-3)) for k, v in times.items()}
    # tree_predict at 1 M rows
    h.set_tree(ref)
    x = torch.as_tensor(np.resize(X, (1 << 20, 39))).cuda()
    h.tree_predict(x)
    torch.cuda.synchronize()
    tp = {}
    for name, tree in (("tree_ref", ref), ("tree_deep", deep)):
        h.set_tree(tree)
        h.tree_predict(x)
        ts = []
        for _ in range(20):
            e0.record()
            h.tree_predict(x)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        tp[name] = dict(ms_median=float(np.median(ts)), rows_per_s=x.shape[0] / (float(np.median(ts)) * 1e-3))
    # banks
    banks = {}
    n = 4096
    chunk = rng.integers(-3000, 3000, size=(n, 160)).astype(np.int16)
    packets = [rng.integers(-3000, 3000, size=480).astype(np.int16) for _ in range(n)]
    for name, cls in (("ffn", None), ("tree_ref", ref)):
        hb = runtime.Handle(0, ffn_weights=w)
        if cls is not None:
            hb.set_tree(cls)
        for kind in ("fixed", "ragged"):
            b = StreamBank(n, handle=hb, max_feed_samples=480 if kind == "ragged" else None)
            ts = []
            for it in range(230):
                t0 = time.perf_counter()
                if kind == "fixed":
                    b.feed(chunk)
                else:
                    b.feed_samples(packets)
                if it >= 30:
                    ts.append((time.perf_counter() - t0) * 1e3)
            banks["%s_%s" % (kind, name)] = dict(p50_ms=float(np.percentile(ts, 50)), p99_ms=float(np.percentile(ts, 99)))
    rec = dict(gpu=gpu_info(), hours=a.hours, reps=a.reps,
               trees=dict(ref=dict(nodes=int(ref.tree_.node_count), depth=int(ref.tree_.max_depth)),
                          deep=dict(nodes=int(deep.tree_.node_count), depth=int(deep.tree_.max_depth))),
               fused=fused, tree_predict=tp, banks=banks)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(rec, f)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
