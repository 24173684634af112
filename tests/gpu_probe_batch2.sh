#!/bin/bash
# round-2 probe batch 2: full suite with fused attention (hard timeouts), then measurements
timeout -s KILL 300 python -m pytest tests/test_attention_gpu.py -q --tb=short 2>&1 | tail -15
echo "attention rc=${PIPESTATUS[0]}"
timeout -s KILL 900 python -m pytest tests -m gpu -q --tb=short --deselect tests/test_attention_gpu.py --durations=12 2>&1 | tail -60
echo "suite rc=${PIPESTATUS[0]}"
bash tests/gpu_round2_ab.sh
