#!/bin/bash
# A/B of the seed-stage probe's first-level bitmap and bulk-copy tile on the c2 step (resident + e2e ms per step)
mkdir -p gpurun_out
run() { name=$1; shift; env "$@" timeout 300 python bench.py --steps 8 --warmup 3 --no-cpu-baseline > gpurun_out/ab_$name.json 2> gpurun_out/ab_$name.err; python -c "
import json; d=json.load(open('gpurun_out/ab_$name.json')); print('$name', round(d['ms_per_step'],2), 'e2e', round(d['e2e']['ms_per_step'],2), 'seed_ms', round(d['roofline_seed']['kernel_ms_per_step'],2), d['step_ms']['resident'])"; }
run all X=1
run nobitmap DMND_NO_BITMAP=1
run nobulk DMND_NO_BULK=1
run none DMND_NO_BITMAP=1 DMND_NO_BULK=1
