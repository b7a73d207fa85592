"""Speech segments and speech audio (vad_segments.cuh) against the fused VAD of the same resident batch.

Workload: N x 10 s utterances in device memory (default 36,000: 3.6e7 label rows, 11.5 GB of PCM, far beyond L2),
segment parameters 250 / 100 / 30 ms.  Label inputs: the fused VAD's own labels, and Markov-run labels (mean run 50
rows).  CUDA events around many launches after warm-up time the fused VAD, the segments call and the gather; the
gather's bytes (speech samples read + written) are set against 7.7 TB/s of HBM3e.  The card's name and power limit
are read in the same run.

    python tools/bench_segments.py [--utts 36000] [--iters 20] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BPS = 7.7e12


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, text=True, timeout=60).stdout.strip().splitlines()[0]
        return [x.strip() for x in q.split(",")]
    except Exception as e:  # noqa: BLE001 -- the numbers still stand, without the card line
        return ["unknown (%s)" % e, "", ""]


def markov_labels(torch, n, mean_run, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    k = int(n / mean_run * 1.2) + 16
    runs = torch.empty(k, device="cuda").exponential_(1.0 / mean_run, generator=g).ceil().long()
    vals = (torch.arange(k, device="cuda") % 2).to(torch.uint8)
    return torch.repeat_interleave(vals, runs)[:n].contiguous()


def timed(torch, fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=36000)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_segments needs a CUDA device")
    from oracle import ref_math as rm
    from vad_b200 import batch, runtime
    from vad_b200.runtime import _ptr
    name, power, sm_clock = card()
    h = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    n_samp = int(args.seconds * 16000)
    offsets, lengths, stride = batch.uniform_layout(args.utts, n_samp)
    pcm = h.synth_pcm(args.utts, n_samp, seed=1234, utt_stride=stride)
    plan = runtime.Plan(h, offsets, lengths, runtime.MODE_VAD)
    rows = plan.total_rows
    labels = torch.empty(rows, dtype=torch.uint8, device="cuda")
    t_vad = timed(torch, lambda: plan.vad(pcm, labels=labels), args.iters)
    S, G, P = (runtime.speech_ms_to_rows(v) for v in (250, 100, 30))
    mx = int(h.lib.vadb200_plan_max_speech_segments(plan._p))
    nb = int(h.lib.vadb200_plan_speech_workspace_bytes(plan._p))
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    segs = torch.empty((mx, 2), dtype=torch.int64, device="cuda")
    so = torch.empty(plan.n_utt + 1, dtype=torch.int64, device="cuda")
    sp = torch.empty(plan.n_utt + 1, dtype=torch.int64, device="cuda")
    out = torch.empty(rows * 160 + 8, dtype=torch.int16, device="cuda")
    st = h.stream
    res = {"what": "speech segments + gather vs fused VAD, resident batch", "gpu": name, "power_limit": power,
           "max_sm_clock": sm_clock, "utterances": args.utts, "seconds_each": args.seconds, "rows": rows,
           "pcm_bytes": int(pcm.numel()) * 2, "params_ms": [250, 100, 30], "params_rows": [S, G, P],
           "iters": args.iters, "fused_vad_s": t_vad, "inputs": {}}
    plan.vad(pcm, labels=labels)
    torch.cuda.synchronize()
    inputs = {"fused_vad_labels": labels, "markov_mean50": markov_labels(torch, rows, 50, 7)}
    for key, lab in inputs.items():
        def seg_call(lab=lab, smoothed=None):
            rc = h.lib.vadb200_plan_speech_segments(plan._p, _ptr(lab), S, G, P, _ptr(smoothed), _ptr(segs), _ptr(so),
                                                    _ptr(sp), _ptr(ws), nb, st)
            assert rc == 0

        def gather_call():
            rc = h.lib.vadb200_plan_gather_speech(plan._p, _ptr(pcm), pcm.numel(), _ptr(segs), _ptr(so), _ptr(sp),
                                                  _ptr(out), out.numel(), st)
            assert rc == 0
        t_seg = timed(torch, seg_call, args.iters * 5)
        seg_call()
        torch.cuda.synchronize()
        speech = int(sp[-1].item())
        k = int(so[-1].item())
        t_gat = timed(torch, gather_call, args.iters)
        moved = 4 * speech                       # int16 read + write per speech sample
        res["inputs"][key] = {
            "speech_fraction": speech / (160.0 * rows), "segments": k,
            "segments_s": t_seg, "segments_share_of_fused_vad": t_seg / t_vad,
            "gather_s": t_gat, "gather_bytes": moved, "gather_bytes_per_s": moved / t_gat,
            "gather_share_of_7p7TBps": moved / t_gat / HBM_BPS}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
