"""Timing experiment: clock64() stamps of CTA 0's tensor-core block phases (not part of the product API).
Needs the hook build:  python -m vad_b200.build --debug-hooks && VADB200_LIB=$PWD/vad_b200/libvadb200_dbg.so python tools/dbg_block_phase.py [tc16|tc]
tc16 (default): the two-tile fp16 block phase (256 frames); tc: the one-tile tf32 block phase (128 frames).
VADB200_DEBUG_SKIP=256 keeps the fp16 issuer from issuing tile 1 (one MMA chain instead of two; labels are garbage)."""
import ctypes as C, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vad_b200 import batch, runtime
impl = sys.argv[1] if len(sys.argv) > 1 else "tc16"
h = runtime.Handle(0, ffn_weights=runtime.glorot_ffn(0))
h.set_ffn_impl(impl)
fn = h.lib.vadb200_debug_timestamps; fn.argtypes = [C.c_void_p]; fn.restype = C.c_int
n_utt, L = 20000, 160000
off, ln, stride = batch.uniform_layout(n_utt, L)
pcm = h.synth_pcm(n_utt, L, utt_stride=stride)
plan = runtime.Plan(h, off, ln, runtime.MODE_VAD)
for _ in range(2): plan.vad(pcm)
buf = torch.zeros(64 * 16, dtype=torch.int64, device=h.device)
fn(C.c_void_p(buf.data_ptr())); plan.vad(pcm); torch.cuda.synchronize(); fn(C.c_void_p(0))
ts = buf.cpu().numpy().reshape(64, 16)
d = np.diff(ts, axis=1)[8:56]
# stamp 1 follows the window features (tc16: and the layer-1 operand store; tc: the store comes after it)
names = ["features (+ A1 store)", "(A1 store +) blob wait", "wait_st+bar", "issue L1", "MMA L1 wait", "epi1",
         "bar+issue L2", "MMA L2 wait", "epi2", "bar+issue L3", "MMA L3 wait", "epi3", "bar+issue L4", "MMA L4 wait",
         "final ld"]
print("%s, VADB200_DEBUG_SKIP=%s: median cycles per stage (CTA 0, thread 0 = the MMA issuer):"
      % (impl, os.environ.get("VADB200_DEBUG_SKIP", "0")))
for n, v in zip(names, np.median(d, axis=0)): print("  %-22s %8.0f" % (n, v))
tot = np.median(ts[8:56, 15] - ts[8:56, 0])
chain = np.median(ts[8:56, 15] - ts[8:56, 3])
print("MMA chain + epilogues (stamp 3 -> 15)", chain)
print("total block phase", tot, "period between block phases", np.median(np.diff(ts[8:56, 0])))
