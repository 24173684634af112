#!/bin/bash
timeout -s KILL 300 python -m pytest tests/test_kernels_gpu.py tests/test_unet_gpu.py tests/test_baseline_shapes_gpu.py -q --tb=short -x 2>&1 | tail -12
for v in "" "FDX_NO_SIDE=1"; do
  echo "== bench c2 $v"
  env $v timeout -s KILL 200 python bench.py --workload c2 --no-sample --no-cpu-baseline --steps 20 2>/dev/null | python -c "
import sys,json
d=json.loads(sys.stdin.read().strip().split('\n')[-1]); print(round(d['value'],1), round(d['ms_per_step'],3), 'e2e', round(d['e2e']['ms_per_step'],3), d['clocks']['sm_mhz'])"
done
for v in ""; do
  echo "== bench c3 $v"
  env $v timeout -s KILL 300 python bench.py --workload c3 --no-sample --no-cpu-baseline --steps 8 2>/dev/null | python -c "
import sys,json
d=json.loads(sys.stdin.read().strip().split('\n')[-1]); print(round(d['value'],1), round(d['ms_per_step'],3), 'e2e', round(d['e2e']['ms_per_step'],3), d['clocks']['sm_mhz'])"
done
