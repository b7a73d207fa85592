#!/usr/bin/env python
"""bench.py -- audio-seconds/second of the fused MFCC+FFN VAD hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (configs[2]): 1,000 h of synthetic 16 kHz int16 audio PER GPU as 360,000 x 10 s
utterances, generated on the device (counter-based integer generator, bit-identical to
vad_b200/synth.py) and resident in HBM (115.2 GB >> 126 MB L2) when the timed region starts.
One step = one pass of the fused kernel over the rank's whole shard -> one uint8 label per
output frame.  Utterances are independent, so ranks share nothing: weak scaling, no collective
on the data path (only the timing all-reduce).

Rank 0 prints ONE JSON line: value (device-resident, CUDA events, max over ranks), e2e (same
metric through the C ABI's host-buffer entry point vadb200_vad_host: pinned host PCM -> H2D ->
kernel -> D2H labels, every step), roofline (algorithmic FP32 flop / kernel time against a live
FMA microbenchmark; HBM fraction alongside), cpu_baseline (the reference-shaped CPU port on the
host cores, bounded sample), clocks and launch count.

--dump-outputs DIR saves what the timed launches returned in their last step (a fixed, seeded sample of whole
utterances' labels) so that two builds can be compared output for output on identical inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the source tree, which may be read-only

METRIC = "audio_seconds_per_second"
UNIT = "audio-s/s"
FLOP_PER_FRAME_FUSED = 24663   # SURVEY.md 8(d): FFT 11520 + power 768 + mel 888 + log 26 + DCT 676 + window 340 + FFN 10208 + 237
FLOP_PER_FRAME_MFCC = 13878    # MFCC-only subtotal (cfg2); dataset rows add 39 (cfg5)
BYTES_PER_FRAME_FUSED = 321    # 160 int16 in + 1 label out
FP32_NOMINAL_TFLOPS = 74.4     # 148 SM x 128 lanes x 2 x 1.965 GHz (fallback denominator)
# dram__bytes_read.sum + dram__bytes_write.sum of fused_kernel<2,2> from the committed `ncu --set full`
# capture (profiles/r3_fused_kernel_2_2_ncu_raw.csv: 5.8241 GB + 0.0227 GB for 17.874 M frames)
NCU_DRAM_BYTES_PER_FRAME = (5.824133e9 + 22.738688e6) / 17874000.0
DUMP_LABEL_BYTES = 48 << 20    # --dump-outputs: float32 labels of as many sampled utterances as fit (64 MB cap in all)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--hours-per-gpu", type=float, default=1000.0)
    ap.add_argument("--utt-seconds", type=float, default=10.0)
    ap.add_argument("--e2e-window-utts", type=int, default=6000, help="utterances per pinned host window (1.92 GB)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-utts-per-core", type=int, default=16)
    ap.add_argument("--ffn-impl", default="tc16", choices=["tc16", "tc", "fp32"],
                    help="FFN contraction: tcgen05 on fp16 hi/lo operands (default), tcgen05 on tf32 hi/lo operands, "
                         "or FP32 CUDA cores")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--stream-ticks", type=int, default=10000)
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the cfg2 / cfg4 / cfg5 sub-records")
    ap.add_argument("--parity-utts", type=int, default=4)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, save the last step's labels of a fixed seeded sample of utterances "
                         "as DIR/labels.npy (float32 [utterances, rows]) and their indices as DIR/utterances.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs saves the GPU path's outputs (--impl ours)")
    return a


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, pw, reasons = [], [], [], set()
        for t, line in self.rows:
            if t < t0 or t > t1 + 0.05:
                continue
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); pw.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw), "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------- CPU arm
def run_cpu_port(utts, procs, steps, warmup, utt_seconds, seed):
    cmd = [sys.executable, "-m", "oracle.cpu_bench", "--utts", str(utts), "--procs", str(procs), "--steps", str(steps),
           "--warmup", str(warmup), "--utt-seconds", str(utt_seconds), "--seed", str(seed)]
    env = dict(os.environ, OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1",
               PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=1500)
    if out.returncode != 0:
        raise RuntimeError("cpu_bench failed: " + out.stderr[-400:])
    return json.loads(out.stdout.strip().splitlines()[-1])


CPU_KIND_NOTE = {
    "reference": "; UNMODIFIED reference process_file (wav read, framing, per-frame mfcc.get_mfcc, ring, deltas) from "
                 "oracle/_ref through the python-3 shim + the oracle's vectorised classifier stage (the reference never "
                 "runs its FFN)",
    "port": "; oracle/ref_loop.py per-frame port (oracle/_ref not staged on this box)",
}


def reference_arm(a):
    """The reference's own CPU implementation of the path on all host cores with its Pool.map shape
    (dataset_creator.py:63-65): the unmodified sources staged under oracle/_ref (kind "reference"), or the
    per-frame port oracle/ref_loop.py where they are absent (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    utts = a.cpu_utts_per_core * cores
    r = run_cpu_port(utts, cores, a.steps, a.warmup, a.utt_seconds, a.seed)
    sample = "%d x %.0f s synthetic utterances per step (%.0f audio-s), Pool(%d)" % (utts, a.utt_seconds,
                                                                                     utts * a.utt_seconds, cores)
    kind = r.get("kind", "port")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["audio_s_per_s"], "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(a, a.gpus, sample_note="bounded sample per step: " + sample),
        "cpu_baseline": {"value": r["audio_s_per_s"], "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": sample + CPU_KIND_NOTE[kind]},
        "e2e": {"value": r["audio_s_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(a, n, sample_note=None):
    c = {"workload": "cfg3: fused MFCC+FFN VAD (39-64-32-16-3, seeded Glorot weights) over %.0f h of synthetic 16 kHz "
                     "int16 audio per GPU, %.0f s utterances, batch-sharded" % (a.hours_per_gpu, a.utt_seconds),
         "hours_per_gpu": a.hours_per_gpu, "total_hours": a.hours_per_gpu * n, "utt_seconds": a.utt_seconds,
         "frame": 400, "hop": 160, "n_fft": 512, "n_mel": 26, "n_ceps": 13, "parallelism": "dp%d (no collective)" % n,
         "l2": "inputs larger than L2 (no flush needed)"}
    if sample_note:
        c["note"] = sample_note
    return c


# ----------------------------------------------------------------------------------------- helpers
def bind_to_gpu_numa(local):
    """Pin this rank's host threads to the CPUs of its GPU's NUMA node BEFORE any pinned allocation, so the e2e
    staging windows are placed next to the PCIe root the GPU hangs off.  Returns a short description."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        if node < 0:
            return {"pci": bdf, "numa_node": node, "bound": False, "why": "platform reports no NUMA affinity"}
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        n_nodes = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")])
        if allowed and n_nodes > 1:
            os.sched_setaffinity(0, allowed)
        return {"pci": bdf, "numa_node": node, "numa_nodes": n_nodes, "cpus": len(allowed),
                "bound": bool(allowed and n_nodes > 1)}
    except Exception as ex:  # sysfs absent (containers): keep going unbound
        return {"bound": False, "why": str(ex)[:80]}


def cuda_time_ms(fn, steps, warmup, torch):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def parity_sample(h, plan, pcm, labels, n_utt, L, stride, seed, first_utt, k):
    """Outside the timed region: k utterances of the RESIDENT shard (first, last, evenly spaced) -- the device PCM
    must equal the host generator bit for bit, and the labels the timed launches produced must equal the oracle's
    on every decisive row; a small re-run of the same utterances with logits checks the logit tolerance."""
    import numpy as np
    from oracle import ref_math as rm
    from vad_b200 import batch, runtime
    from vad_b200.synth import synth_utterance
    w = runtime.glorot_ffn(0)
    idx = sorted(set(int(round(i * (n_utt - 1) / max(k - 1, 1))) for i in range(k)))
    ro = plan.row_offsets
    ok_pcm = ok_lab = ok_logit = True
    max_err = 0.0
    sub = []
    for u in idx:
        host = synth_utterance(seed, first_utt + u, L)
        dev = pcm[u * stride:u * stride + L].cpu().numpy()
        ok_pcm &= bool(np.array_equal(host, dev))
        sub.append(host)
        _, feats, ref_logits, ref_labels = rm.vad_utterance(host, w)
        got = labels[int(ro[u]):int(ro[u + 1])].cpu().numpy()
        fin = np.isfinite(feats).all(axis=1)
        srt = np.sort(ref_logits[fin], axis=1)
        dec = (srt[:, -1] - srt[:, -2]) > 2 * (1e-3 + 1e-3 * np.abs(srt[:, -1]))
        ok_lab &= bool(np.array_equal(got[fin][dec], ref_labels[fin][dec]) and np.all(got[~fin] == 0))
    la, lo = batch.vad_batch(sub, handle=h, want_logits=True)
    for host, lg in zip(sub, lo):
        _, feats, ref_logits, _ = rm.vad_utterance(host, w)
        fin = np.isfinite(feats).all(axis=1)
        err = np.abs(lg.cpu().numpy()[fin] - ref_logits[fin])
        max_err = max(max_err, float(err.max()) if err.size else 0.0)
        ok_logit &= bool(np.all(err <= 1e-3 + 1e-3 * np.abs(ref_logits[fin])))
    return {"result": "pass" if (ok_pcm and ok_lab and ok_logit) else "fail", "utterances": idx,
            "pcm_bit_identical_to_host_generator": ok_pcm, "labels_equal_oracle_on_decisive_rows": ok_lab,
            "logits_within_1e-3": ok_logit, "max_logit_abs_err": max_err,
            "oracle": "oracle/ref_math.py (float64 restatement pinned to the reference's golden vectors)"}


def dump_outputs(out_dir, plan, labels, n_utt, torch):
    """The labels the timed launches wrote in their last step, for whole utterances drawn with a fixed seed (the
    same utterances for the same arguments, whatever the build): DIR/labels.npy float32 [k, rows per utterance] and
    DIR/utterances.npy float64 [k], the utterances' indices in the rank-0 shard."""
    import numpy as np
    ro = plan.row_offsets
    rows = int(ro[1] - ro[0])                                   # uniform layout: every utterance has as many rows
    k = min(n_utt, DUMP_LABEL_BYTES // (4 * max(rows, 1)))
    utts = np.sort(np.random.default_rng(0).choice(n_utt, size=k, replace=False))
    idx = torch.from_numpy(ro[utts][:, None] + np.arange(rows)).to(labels.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "labels.npy"), labels[idx].float().cpu().numpy())
    np.save(os.path.join(out_dir, "utterances.npy"), utts.astype(np.float64))


def stream_record(h, a, torch):
    """configs[3]: a.streams concurrent 16 kHz streams in 10 ms chunks through analyser.StreamBank (one CUDA-graph
    launch per tick: H2D of the chunks, stream_feed_kernel, D2H of the labels).  Latency = host wall clock from
    'chunk batch is in pinned host memory' to 'labels are readable on the host', per tick."""
    import numpy as np
    from vad_b200.analyser import StreamBank
    bank = StreamBank(a.streams, handle=h)
    rng = np.random.default_rng(0)
    pool = torch.from_numpy((rng.standard_normal((32, a.streams, 160)) * 3000).astype(np.int16))
    warm = 100
    lat = np.zeros(a.stream_ticks)
    speech = 0
    for t in range(warm + a.stream_ticks):
        bank.h_chunks.copy_(pool[t % 32])            # the tick's audio arrives in pinned memory
        t0 = time.perf_counter()
        labels = bank.feed_pinned()
        dt = time.perf_counter() - t0
        if t >= warm:
            lat[t - warm] = dt
            speech += int((labels == 1).sum())
    ms = np.sort(lat) * 1e3
    p99 = float(ms[int(len(ms) * 0.99)])
    return {"metric": "stream_chunk_latency_ms", "streams": a.streams, "ticks": a.stream_ticks, "warmup_ticks": warm,
            "chunk_ms": 10.0, "cuda_graph": bool(bank.use_graph and bank._graphs), "launches_per_tick": 1,
            "p50_ms": float(ms[len(ms) // 2]), "p99_ms": p99, "max_ms": float(ms[-1]), "mean_ms": float(ms.mean()),
            "keeps_up_with_realtime": bool(p99 < 10.0), "realtime_headroom_at_p99": 10.0 / p99,
            "audio_s_per_s_at_mean": float(a.streams * 0.010 / (ms.mean() * 1e-3)), "speech_decisions": speech,
            "algorithmic_lag_frames": 3, "h2d_bytes_per_tick": a.streams * 320, "d2h_bytes_per_tick": a.streams,
            "timing": "host wall clock around StreamBank.feed_pinned() (graph launch + stream sync), rank 0"}


def analyser_record(h, torch):
    """FusedAnalyser.feed_frame (the single-stream SKLearnAnalyzer drop-in): p50 / p99 per call."""
    import numpy as np
    from vad_b200.analyser import FusedAnalyser
    from vad_b200.synth import synth_utterance
    an = FusedAnalyser(handle=h)
    pcm = synth_utterance(5, 0, 400 * 1205).astype(np.float32).reshape(1205, 400)
    an.load_init_inactive_frames(list(pcm[:5]))
    lat = []
    for i in range(1205):
        t0 = time.perf_counter()
        an.feed_frame(pcm[i])
        dt = time.perf_counter() - t0
        if i >= 205:
            lat.append(dt)
    ms = np.sort(np.array(lat)) * 1e3
    return {"calls": len(lat), "p50_ms": float(ms[len(ms) // 2]), "p99_ms": float(ms[int(len(ms) * 0.99)]),
            "max_ms": float(ms[-1]), "frame_ms": 25.0,
            "note": "per call: one MFCC-frame launch, one window-classify launch, one D2H sync"}


def cfg2_record(h, peak, hbm_peak, torch):
    """configs[1]: MFCC-only, 1024 x 10 s (327.68 MB in, 53.1 MB out; inputs larger than L2)."""
    from vad_b200 import batch, runtime
    n_utt, L = 1024, 160000
    off, ln, stride = batch.uniform_layout(n_utt, L)
    pcm = h.synth_pcm(n_utt, L, seed=0, first_utt=0, utt_stride=stride)
    plan = runtime.Plan(h, off, ln, runtime.MODE_MFCC)
    out = torch.empty((plan.total_rows, 13), dtype=torch.float32, device=h.device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=h.device)
    for _ in range(3):
        plan.mfcc(pcm, out=out)
    tot = 0.0
    for _ in range(10):
        flush.fill_(1)                                 # evict the input's tail from the 126 MB L2
        tot += cuda_time_ms(lambda: plan.mfcc(pcm, out=out), 1, 0, torch)
    ms = tot / 10
    frames = plan.total_rows
    ach = frames * FLOP_PER_FRAME_MFCC / (ms * 1e-3) / 1e12
    gbs = frames * (320 + 52) / (ms * 1e-3) / 1e9
    return {"workload": "cfg2: MFCC-only, 1024 x 10 s utterances", "value": n_utt * 10.0 / (ms * 1e-3), "unit": UNIT,
            "ms_per_step": ms, "frames": int(frames), "segment_frames": plan.segment_frames,
            "l2": "256 MB flush buffer written between timed launches",
            "roofline": {"bound": "fp32", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                         "kernel": "fused_kernel<0,0>", "algorithmic_flop_per_frame": FLOP_PER_FRAME_MFCC,
                         "hbm": {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                                 "algorithmic_bytes_per_frame": 372}}}


def cfg5_record(h, peak, hbm_peak, torch):
    """configs[4]: 8192 ragged 2-30 s utterances (seed 7), deltas + delta-deltas (39-dim rows), packed offsets."""
    import numpy as np
    from vad_b200 import runtime
    n_utt, smax = 8192, 480000
    rng = np.random.default_rng(7)
    lens = rng.integers(32000, smax + 1, size=n_utt).astype(np.int64)
    off = np.arange(n_utt, dtype=np.int64) * smax                 # 8-sample-aligned offsets (gaps are never read)
    pcm = h.synth_pcm(n_utt, smax, seed=7, first_utt=0, utt_stride=smax)
    dplan = runtime.Plan(h, off, lens, runtime.MODE_DATASET)
    vplan = runtime.Plan(h, off, lens, runtime.MODE_VAD)
    rows = torch.empty((dplan.total_rows, 39), dtype=torch.float32, device=h.device)
    labels = torch.empty((vplan.total_rows,), dtype=torch.uint8, device=h.device)
    ms_rows = cuda_time_ms(lambda: dplan.mfcc(pcm, out=rows), 5, 3, torch)
    ms_vad = cuda_time_ms(lambda: vplan.vad(pcm, labels=labels), 5, 3, torch)
    audio_s = float(lens.sum()) / 16000.0
    fr = dplan.total_rows
    ach = fr * (FLOP_PER_FRAME_MFCC + 39) / (ms_rows * 1e-3) / 1e12
    gbs = fr * (320 + 156) / (ms_rows * 1e-3) / 1e9
    achv = fr * FLOP_PER_FRAME_FUSED / (ms_vad * 1e-3) / 1e12
    return {"workload": "cfg5: 8192 ragged utterances, 2-30 s uniform (seed 7), 39-dim dataset rows, packed",
            "audio_hours": audio_s / 3600.0, "rows": int(fr), "segment_frames": dplan.segment_frames,
            "value": audio_s / (ms_rows * 1e-3), "unit": UNIT, "ms_per_step": ms_rows,
            "l2": "inputs larger than L2 (4.2 GB of PCM read per launch)",
            "roofline": {"bound": "fp32", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                         "kernel": "fused_kernel<1,0>", "algorithmic_flop_per_frame": FLOP_PER_FRAME_MFCC + 39,
                         "hbm": {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                                 "algorithmic_bytes_per_frame": 476}},
            "vad": {"value": audio_s / (ms_vad * 1e-3), "unit": UNIT, "ms_per_step": ms_vad,
                    "roofline_frac": achv / peak}}


# ----------------------------------------------------------------------------------------- GPU arm
def main():
    a = parse_args()
    if a.impl == "reference":
        reference_arm(a)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs CUDA devices (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from vad_b200 import batch, runtime

    h = runtime.Handle(local, ffn_weights=runtime.glorot_ffn(0))
    h.set_ffn_impl(a.ffn_impl)
    L = int(round(a.utt_seconds * 16000))
    n_utt = int(round(a.hours_per_gpu * 3600.0 / a.utt_seconds))
    offsets, lengths, stride = batch.uniform_layout(n_utt, L)
    need = n_utt * stride * 2 + n_utt * 1000 + (3 << 30)
    free, _ = torch.cuda.mem_get_info(dev)
    if need > free:  # never drive the box out of memory: shrink and say so
        if a.dump_outputs:
            raise SystemExit("--dump-outputs: %.0f h per GPU do not fit in free GPU memory; a smaller workload's "
                             "outputs would not compare with a full run's" % a.hours_per_gpu)
        n_utt = int((free - (4 << 30)) // (stride * 2 + 1000))
        offsets, lengths, stride = batch.uniform_layout(n_utt, L)
        a.hours_per_gpu = n_utt * a.utt_seconds / 3600.0
    pcm = torch.empty(n_utt * stride + 8, dtype=torch.int16, device=dev)
    pcm[-8:].zero_()
    h.synth_pcm(n_utt, L, seed=a.seed, first_utt=rank * n_utt, utt_stride=stride, out=pcm)
    plan = runtime.Plan(h, offsets, lengths, runtime.MODE_VAD)
    labels = torch.empty(plan.total_rows, dtype=torch.uint8, device=dev)
    audio_s = n_utt * a.utt_seconds
    frames = plan.total_rows
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- device-resident timing ---------------------------------------------------------------------
    for _ in range(max(a.warmup, 3)):
        plan.vad(pcm, labels=labels)
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = h.lib.vadb200_launch_count()
    t_w0 = time.perf_counter()
    e0.record()
    for _ in range(a.steps):
        plan.vad(pcm, labels=labels)
    e1.record()
    torch.cuda.synchronize()
    t_w1 = time.perf_counter()
    barrier()
    launches = h.lib.vadb200_launch_count() - launches0
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if sampler:
        time.sleep(0.1)
        sampler.stop()
    ms_per_step = ms_total / a.steps
    if rank == 0 and a.dump_outputs:
        dump_outputs(a.dump_outputs, plan, labels, n_utt, torch)
    total_audio = sum_over_ranks(audio_s)
    value = total_audio / (ms_per_step * 1e-3)
    speech_frac = float(labels[: min(frames, 50_000_000)].float().mean().item())
    parity = None
    if rank == 0 and a.parity_utts > 0:
        parity = parity_sample(h, plan, pcm, labels, n_utt, L, stride, a.seed, rank * n_utt, a.parity_utts)

    # ---- end to end through the host-buffer C-ABI entry point ---------------------------------------
    e2e = None
    if not a.no_e2e:
        win = min(a.e2e_window_utts, n_utt)
        while n_utt % win:
            win -= 1
        n_win = n_utt // win
        w_off, w_len, _ = batch.uniform_layout(win, L)
        wplan = runtime.Plan(h, w_off, w_len, runtime.MODE_VAD)
        h_pcm = torch.empty(win * stride + 8, dtype=torch.int16).pin_memory()
        h_pcm.copy_(pcm[: win * stride + 8])
        h_lab = torch.empty(wplan.total_rows, dtype=torch.uint8).pin_memory()
        torch.cuda.synchronize()
        wplan.vad_host(h_pcm, labels_host=h_lab)                       # warm-up + sanity: same labels as the device path
        same = bool(torch.equal(h_lab, labels[: wplan.total_rows].cpu()))
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.e2e_steps):
            for _w in range(n_win):
                wplan.vad_host(h_pcm, labels_host=h_lab)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        barrier()
        # the host's concurrent H2D ceiling: every rank copies its pinned window, no kernel, between barriers
        d_win = torch.empty(win * stride + 8, dtype=torch.int16, device=dev)
        d_win.copy_(h_pcm, non_blocking=True)
        torch.cuda.synchronize()
        barrier()
        t0c = time.perf_counter()
        reps = 8
        for _ in range(reps):
            d_win.copy_(h_pcm, non_blocking=True)
        torch.cuda.synchronize()
        dtc = max_over_ranks(time.perf_counter() - t0c)
        barrier()
        ceil_gbs = sum_over_ranks(reps * h_pcm.numel() * 2) / dtc / 1e9
        del d_win
        e2e_gbs = sum_over_ranks(n_win * win * stride * 2) * a.e2e_steps / dt / 1e9
        e2e = {"value": total_audio * a.e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(sum_over_ranks(n_win * win * stride * 2)),
               "d2h_bytes_per_step": int(sum_over_ranks(n_win * wplan.total_rows)),
               "ms_per_step": 1e3 * dt / a.e2e_steps, "timing": "host wall clock around blocking C-ABI calls, max over ranks",
               "host_window_bytes": int(win * stride * 2), "windows_per_step": n_win, "labels_match_device_path": same,
               "h2d_GBps": e2e_gbs, "h2d_ceiling_GBps": ceil_gbs, "frac_of_h2d_ceiling": e2e_gbs / ceil_gbs,
               "h2d_ceiling_note": "all %d ranks copying their pinned 1.92 GB window concurrently, no kernel "
                                   "(the e2e roofline of this host at this N)" % world,
               "numa": numa}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant (only) kernel -----------------------------------------------------
    peak_reg = h.fp32_peak(0, 2048)
    peak_const = h.fp32_peak(1, 2048)
    peak_x2 = h.fp32_peak(2, 2048)
    peak = max(peak_reg, peak_const, peak_x2)   # the largest of the three is the denominator
    peak_src = "live FMA microbenchmark on this GPU (vadb200_fp32_peak: FFMA reg %.1f / FFMA const-operand %.1f / " \
               "packed FFMA2 %.1f TFLOP/s; the maximum is used); MEASURED_PEAKS.json has no FP32 figure" % (
                   peak_reg, peak_const, peak_x2)
    if not peak or peak <= 0:
        peak, peak_src = FP32_NOMINAL_TFLOPS, "nominal fallback 148x128x2x1.965 GHz"
    hbm_peak = None
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            hbm_peak = float(json.load(f)["hbm_gbs"])
    except Exception:
        hbm_peak = 6650.0
    kern_s = ms_per_step * 1e-3                     # one fused_kernel<VAD> launch per step
    achieved = frames * FLOP_PER_FRAME_FUSED / kern_s / 1e12
    hbm_ach = frames * BYTES_PER_FRAME_FUSED / kern_s / 1e9
    roofline = {"bound": "fp32", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": frames * NCU_DRAM_BYTES_PER_FRAME if a.ffn_impl != "fp32" else None,
                "traffic_note": "bytes per launch = frames x %.1f B/frame from the ncu capture in profiles/ (r3) " % NCU_DRAM_BYTES_PER_FRAME +
                                "(algorithmic 321 B/frame: no re-reads)",
                "kernel": "%s (MFCC+FFN VAD, FFN on %s)" % (
                    {"tc16": "fused_kernel<2,2>", "tc": "fused_kernel<2,1>", "fp32": "fused_kernel<2,0>"}[a.ffn_impl],
                    {"tc16": "tcgen05 kind::f16, statically scaled fp16 hi/lo operands",
                     "tc": "tcgen05 kind::tf32, hi/lo operands", "fp32": "FP32 CUDA cores"}[a.ffn_impl]),
                "launches_per_step": 1,
                "algorithmic_flop_per_frame": FLOP_PER_FRAME_FUSED, "frames_per_launch": int(frames),
                "peak_source": peak_src, "nominal_fp32_tflops": FP32_NOMINAL_TFLOPS,
                "frac_of_nominal": achieved / FP32_NOMINAL_TFLOPS,
                "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                        "algorithmic_bytes_per_frame": BYTES_PER_FRAME_FUSED}}

    # ---- CPU baseline next to it (N = 1 only) ---------------------------------------------------------
    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        cores = os.cpu_count() or 1
        utts = a.cpu_utts_per_core * cores
        try:
            r = run_cpu_port(utts, cores, 1, 1, a.utt_seconds, a.seed)
            kind = r.get("kind", "port")
            cpu = {"value": r["audio_s_per_s"], "unit": UNIT, "cores": cores, "kind": kind,
                   "sample": "%d x %.0f s utterances of the same synthetic workload (%.0f audio-s) under "
                             "multiprocessing.Pool(%d)%s" % (utts, a.utt_seconds, utts * a.utt_seconds, cores,
                                                             CPU_KIND_NOTE[kind])}
        except Exception as ex:  # the GPU numbers stand on their own
            cpu = {"value": None, "unit": UNIT, "cores": cores, "kind": "port", "sample": "failed: %s" % ex}

    # ---- the other configs of BASELINE.json, each with its own roofline (rank 0, after every timed region) ----
    extra = {}
    if not a.no_extra_configs:
        del pcm, labels
        torch.cuda.empty_cache()
        try:
            extra["stream"] = stream_record(h, a, torch)
            extra["analyser_feed_frame"] = analyser_record(h, torch)
            extra["cfg2"] = cfg2_record(h, peak, hbm_peak, torch)
            extra["cfg5"] = cfg5_record(h, peak, hbm_peak, torch)
        except Exception as ex:  # the headline line stands on its own
            extra["error"] = repr(ex)[:300]

    clocks = sampler.summary(t_w0, t_w1) if sampler else None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (device-generated counter-based int16 noise with a speech-like on/off envelope; "
                "random-init FFN weights)",
        "config": workload_config(a, world), "e2e": e2e, "gpu_launches": int(sum_over_ranks(launches)) if world == 1 else int(launches * world),
        "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
        "parity_sample": parity, "stream": extra.get("stream"), "analyser_feed_frame": extra.get("analyser_feed_frame"),
        "cfg2": extra.get("cfg2"), "cfg5": extra.get("cfg5"), "extra_error": extra.get("error"),
        "frames_per_step": int(frames * world), "speech_fraction": speech_frac, "ffn_impl": a.ffn_impl,
        "gpu": torch.cuda.get_device_name(local),
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
