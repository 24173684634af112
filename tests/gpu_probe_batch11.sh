#!/bin/bash
# round-2 batch 11: side-input L2 prefetch in the epilogues, column-tile rule for small pixel counts, merged
# GroupNorm-backward finalize, attention with two CTAs / two element-wise warp groups: parity, then A/B numbers.
mkdir -p gpurun_out
timeout -s KILL 900 python -m pytest tests/test_tc_gpu.py tests/test_optin_kernels_gpu.py tests/test_kernels_gpu.py tests/test_attention_gpu.py tests/test_conv1x1_gpu.py -q --tb=short -x 2>&1 | tail -12
timeout -s KILL 600 python -m pytest tests/test_unet_gpu.py -q --tb=short -x 2>&1 | tail -5
for v in "FDX_TC_BN_V1=1" "FDX_X=0"; do
  for m in fwd dgrad; do
    echo "== layers 64 $m $v"; env $v timeout -s KILL 200 python tests/gpu_bench_layers.py 64 256 $m 2>&1 | grep -E " 8x8|16x16|TOTAL"
  done
done
echo "== attention old"; FDX_ATTN_NO_DUAL=1 FDX_ATTN_BWD_EWG1=1 timeout -s KILL 200 python tests/gpu_bench_attention.py 2>&1 | cut -c1-150
echo "== attention new"; timeout -s KILL 200 python tests/gpu_bench_attention.py 2>&1 | cut -c1-150
for v in "FDX_X=0" "FDX_TC_BN_V1=1"; do
  echo "== bench c2 $v"
  env $v FDX_BENCH_CALLS=gpurun_out/calls_c2_$v.txt timeout -s KILL 200 python bench.py --workload c2 --no-cpu-baseline --steps 20 2>/dev/null | python -c "
import sys,json
d=json.loads(sys.stdin.read().strip().split('\n')[-1]); print(round(d['value'],1), round(d['ms_per_step'],3), 'e2e', round(d['e2e']['ms_per_step'],3), 'euler', round(d['sample']['denoise_steps_per_sec'],1), d['clocks']['sm_mhz'], d['launches_per_step'])"
done
echo "== bench c3"
FDX_BENCH_CALLS=gpurun_out/calls_c3.txt timeout -s KILL 300 python bench.py --workload c3 --no-cpu-baseline --no-sample --steps 5 2>/dev/null | python -c "
import sys,json
d=json.loads(sys.stdin.read().strip().split('\n')[-1]); print(round(d['value'],1), round(d['ms_per_step'],3), 'e2e', round(d['e2e']['ms_per_step'],3), d['clocks']['sm_mhz'], d['launches_per_step']); print({k:(round(v['ms'],2),round(v['tflops'])) for k,v in d['roofline']['kernels'].items()})"
