#!/bin/bash
# GPU test driver used during development (gpurun): the new fused-attention kernels first, isolated and under
# a hard timeout (a dead-locked mbarrier wait must not hold the box), then the whole -m gpu suite.
mkdir -p gpurun_out
timeout -s KILL 420 python -m pytest tests/test_attention_gpu.py -q -x 2>&1 | tail -25 > gpurun_out/t_attn.log
rc=${PIPESTATUS[0]}
echo "attention rc=$rc"; tail -25 gpurun_out/t_attn.log
if [ $rc -ne 0 ]; then export FDX_ATTN_UNFUSED=1; echo "== running the rest with FDX_ATTN_UNFUSED=1"; fi
timeout -s KILL 1200 python -m pytest tests -m gpu -q --deselect tests/test_attention_gpu.py 2>&1 | tail -60 > gpurun_out/t_all.log
echo "suite rc=${PIPESTATUS[0]}"; tail -60 gpurun_out/t_all.log
