#!/bin/bash
# round-2 batch 20: GroupNorm apply straight from the epilogue column sums (fdx_groupnorm_apply_cols)
timeout -s KILL 900 python -m pytest tests/test_kernels_gpu.py tests/test_unet_gpu.py tests/test_baseline_shapes_gpu.py tests/test_train_gpu.py tests/test_samplers_gpu.py -q --tb=short -x 2>&1 | tail -5
for v in "FDX_X=0" "FDX_X=1"; do
  echo "== bench c2 $v"
  env $v timeout -s KILL 200 python bench.py --workload c2 --no-cpu-baseline --steps 20 2>/dev/null | python -c "
import sys,json
d=json.loads(sys.stdin.read().strip().split('\n')[-1]); print(round(d['value'],1), round(d['ms_per_step'],3), 'e2e', round(d['e2e']['ms_per_step'],3), 'euler', round(d['sample']['denoise_steps_per_sec'],1), d['clocks']['sm_mhz'], d['launches_per_step'])"
done
