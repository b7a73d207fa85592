#!/bin/bash
# Phase ablations of fused_kernel<2,1> on the hook build (python -m vad_b200.build --debug-hooks):
# VADB200_DEBUG_SKIP mask: 1 FFT, 2 mel, 4 DCT, 8 block phase, 16 blob TMA, 32 MMA issue+waits, 64 window features, 128 epilogues (32 and 128: tf32 tile only), 256 no second fp16 tile (MMA chain of one tile).
# Prints ms per 1000 h for each mask (results are garbage under ablation: timing only).
for M in ${@:-0 8 12 14 15 1 2 4 32 64 128}; do
  echo -n "mask $M: "
  VADB200_LIB=$PWD/vad_b200/libvadb200_dbg.so VADB200_DEBUG_SKIP=$M python bench.py --hours-per-gpu 200 --steps 3 --warmup 3 --no-cpu-baseline --no-e2e --no-extra-configs 2>&1 | tail -1 | python -c "import json,sys; d=json.loads(sys.stdin.read()); print(round(d['ms_per_step']*5,2))"
done
