#!/bin/bash
# Resampler-kernel variants on the BASELINE configs[1] workload: prints kernel ms and roofline fraction per setting.
# usage: tools/sweep_kernel.sh "ESPB_PPC=0" "ESPB_PPC=10" ...
mkdir -p gpurun_out
for cfg in "$@"; do
  env $cfg python bench.py --steps 10 --warmup 3 --no-e2e --no-cpu-baseline 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); r=d['roofline']
print('$cfg', 'step_ms=%.3f kernel_ms=%.3f frac=%.4f peak=%.1f' % (d['ms_per_step'], r['kernel_ms'], r['frac'], r['peak']))"
done
