#!/bin/bash
# sweep the launch-time knobs of CGRT_TUNE (blocks, chains, coop, waveblocks; speed only, results are identical by construction)
# example: tools/tune_sweep.sh "blocks=6" "blocks=8" "chains=2,coop=30000"
run() { echo -n "CGRT_TUNE=$1 : "; CGRT_TUNE="$1" python bench.py --steps 6 --warmup 3 --no-cpu-baseline 2>&1 | python -c "
import sys,json
for l in sys.stdin:
    if l.startswith('{'):
        j=json.loads(l); print('ms/frame', round(j['ms_per_step'],3), j['config']['kernel_ms_per_frame_rank0'])
"; }
for t in "$@"; do run "$t"; done
