"""The 16 kHz resampler (vad_resample.cuh) on device-resident audio, per source rate.

Workload per rate: 10 s utterances of synthetic int16 PCM (vadb200_synth_pcm) at the source rate, --gb of input in
device memory (default 2 GB: far beyond the 126 MB L2, so every pass reads HBM).  CUDA events around --iters launches
after warm-up time resample_kernel<int16_t>.  Reported per rate: kernel time, output audio seconds per second, the
FMA work (2 K flop per output: K taps of the polyphase row, zero padding included) over the FFMA2 peak that
vadb200_fp32_peak measures in the same run, the HBM traffic (int16 in + out) over 7.7 TB/s, which of the two bounds
the kernel, and resample + fused VAD (MODE_VAD plan on the resampled batch) against the fused VAD alone on the same
16 kHz audio.  The card's name and power limit are read in the same run.

    python tools/bench_resample.py [--gb 2] [--iters 10] [--rates 8000,44100,48000,96000] [--out result.json]
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


def timed(torch, fn, iters, warmup=2):
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
    ap.add_argument("--gb", type=float, default=2.0)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rates", default="8000,44100,48000,96000")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    from oracle import ref_math as rm
    from vad_b200 import runtime
    if not torch.cuda.is_available():
        raise SystemExit("bench_resample needs a CUDA device")
    h = runtime.Handle(0, ffn_weights=rm.glorot_ffn(0))
    peak = h.fp32_peak(2)
    name, power, clock = card()
    results = []
    for rate in [int(r) for r in args.rates.split(",")]:
        r = runtime.Resampler(h, rate)
        utt = 10 * rate
        n_utt = max(1, int(args.gb * 1e9 / 2 / utt))
        pcm = h.synth_pcm(n_utt, utt, seed=rate)
        offs = np.arange(n_utt, dtype=np.int64) * utt
        lens = np.full(n_utt, utt, dtype=np.int64)
        out, o16, l16 = r.run(pcm, offs, lens)
        t_rs = timed(torch, lambda: r.run(pcm, offs, lens, out=out), args.iters)
        n_out = int(l16.sum())
        up, down = r.up, r.down
        n_taps = int(h.lib.vadb200_resample_taps(rate, None))
        K = int(-(-n_taps // up))
        flop = 2.0 * K * n_out
        byts = 2.0 * (n_utt * utt + n_out)
        t_fma, t_mem = flop / (peak * 1e12), byts / HBM_BPS
        plan = runtime.Plan(h, o16, l16, runtime.MODE_VAD)
        labels = torch.empty(plan.total_rows, dtype=torch.uint8, device="cuda")
        t_vad = timed(torch, lambda: plan.vad(out, labels=labels), args.iters)
        t_both = timed(torch, lambda: (r.run(pcm, offs, lens, out=out), plan.vad(out, labels=labels)), args.iters)
        res = {"rate": rate, "up": up, "down": down, "taps_per_output": K, "utterances": n_utt,
               "input_gb": round(n_utt * utt * 2 / 1e9, 3), "resample_ms": round(t_rs * 1e3, 3),
               "output_audio_s_per_s": round(n_out / 16000.0 / t_rs, 1),
               "fp32_tflops": round(flop / t_rs / 1e12, 2), "fp32_peak_tflops": round(peak, 2),
               "share_of_fp32_peak": round(t_fma / t_rs, 3), "hbm_tb_s": round(byts / t_rs / 1e12, 3),
               "share_of_hbm": round(t_mem / t_rs, 3), "bound": "fp32" if t_fma >= t_mem else "hbm",
               "vad_16k_ms": round(t_vad * 1e3, 3), "resample_plus_vad_ms": round(t_both * 1e3, 3),
               "card": name, "power_limit": power, "max_sm_clock": clock}
        print(json.dumps(res), flush=True)
        results.append(res)
        del pcm, out, plan, labels
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
