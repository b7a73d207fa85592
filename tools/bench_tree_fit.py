"""Decision-tree fit on the device (runtime.TreeFitter) against sklearn's on the host, on the reference's training mix.

Workload: device analyser features of synthetic audio (Handle.synth_pcm, 10 s utterances), labelled with the FFN's
decisions with 10 % flipped (like the `ref` tree of tests/test_gpu_tree.py), sampled to 4.5 M speech + 2 M
non-speech rows (decision.res: 4.5 M voiced + 2 M unvoiced frames).  Device: median of --reps synchronised fits at the
reference grid-search hyperparameters (max_depth=25, min_samples_leaf=20, min_samples_split=22) and unbounded (sklearn
defaults), with node count, depth and tied_nodes.  sklearn: one fit at the reference hyperparameters on the first
--sklearn-rows rows (all rows with --sklearn-rows 0), and whether it equals the device's fit of those same rows when
that fit reports tied_nodes == 0.  Prints one JSON record; --out also writes it."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from vad_b200 import runtime  # noqa: E402

REF = dict(max_depth=25, min_samples_leaf=20, min_samples_split=22)


def gpu_info():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                           "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()


def depth_of(t):
    d = np.zeros(t["feature"].shape[0], np.int64)
    for k in range(d.shape[0]):
        if t["children_left"][k] >= 0:
            d[t["children_left"][k]] = d[t["children_right"][k]] = d[k] + 1
    return int(d.max())


def workload(h, speech_rows, other_rows, seed=0):
    utt = 10 * 16000
    rows_per_utt = runtime.outputs_for_length(utt)
    n_utt = int(1.3 * (speech_rows + other_rows) / rows_per_utt) + 1
    xs, ys = [], []
    g = torch.Generator(device="cuda").manual_seed(seed)
    for u0 in range(0, n_utt, 2000):
        k = min(2000, n_utt - u0)
        pcm = h.synth_pcm(k, utt, first_utt=u0)
        offs = np.arange(k, dtype=np.int64) * utt
        plan = runtime.Plan(h, offs, np.full(k, utt, np.int64), runtime.MODE_VAD)
        lab, _, ft = plan.vad(pcm, want_feats=True)
        ok = torch.isfinite(ft).all(dim=1)
        flip = torch.rand(lab.shape, generator=g, device="cuda") < 0.1
        xs.append(ft[ok])
        ys.append((lab ^ flip.to(torch.uint8))[ok])
        plan.close()
    x, y = torch.cat(xs), torch.cat(ys)
    pick = []
    for cls, want in ((1, speech_rows), (0, other_rows)):
        idx = torch.nonzero(y == cls).flatten()
        pick.append(idx[torch.randint(0, idx.numel(), (want,), generator=g, device="cuda")] if idx.numel() < want
                    else idx[torch.randperm(idx.numel(), generator=g, device="cuda")[:want]])
    pick = torch.cat(pick)
    pick = pick[torch.randperm(pick.numel(), generator=g, device="cuda")]
    return x[pick].contiguous(), y[pick].contiguous(), int(x.shape[0])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--speech-rows", type=int, default=4_500_000)
    ap.add_argument("--other-rows", type=int, default=2_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sklearn-rows", type=int, default=250_000, help="0: all rows")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.init()
    h = runtime.Handle(0, ffn_weights=runtime.glorot_ffn(0))
    x, y, made = workload(h, a.speech_rows, a.other_rows)
    n = x.shape[0]
    rec = dict(gpu=gpu_info(), rows=n, speech_rows=a.speech_rows, other_rows=a.other_rows, feature_rows_made=made)
    fitter = runtime.TreeFitter(h, n)
    for name, kw in (("reference", REF), ("unbounded", {})):
        times, t = [], None
        for _ in range(a.reps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            t = fitter.fit(x, y, **kw)
            times.append(time.perf_counter() - t0)
        rec[name] = dict(params=kw, median_s=float(np.median(times[1:])), times_s=times[1:],
                         nodes=int(t["feature"].shape[0]), depth=depth_of(t), tied_nodes=t["tied_nodes"])
        print(name, rec[name], flush=True)
    m = n if a.sklearn_rows <= 0 else min(n, a.sklearn_rows)
    from sklearn.tree import DecisionTreeClassifier
    import _ref_tree_fit as R
    X, Y = x[:m].cpu().numpy(), y[:m].cpu().numpy().astype(np.int64)
    t0 = time.perf_counter()
    clf = DecisionTreeClassifier(random_state=0, **REF).fit(X, Y)
    sk_s = time.perf_counter() - t0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev = fitter.fit(x[:m].contiguous(), y[:m].contiguous(), **REF)
    dev_s = time.perf_counter() - t0
    rec["sklearn"] = dict(rows=m, subsampled=m < n, fit_s=sk_s, host_cpus=os.cpu_count(), device_fit_s=dev_s,
                          nodes=int(clf.tree_.node_count), device_tied_nodes=dev["tied_nodes"],
                          equal=bool(R.same_tree(dev, R.sklearn_arrays(clf))))
    rec["gpu_after"] = gpu_info()
    print(json.dumps(rec))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
