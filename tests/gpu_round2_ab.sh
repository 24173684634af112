#!/bin/bash
# Round-2 A/B micro-benchmarks: new weight-gradient kernel vs the round-1 kernels, the two-pass GroupNorm
# backward, fused attention.  Outputs: <dir>/layers_r02_*.txt, <dir> = the first argument (default: a directory
# under $TMPDIR, so that nothing is written into the source tree).
out=${1:-${TMPDIR:-/tmp}/fdx_round2_ab}
mkdir -p "$out"
timeout 300 python tests/gpu_bench_layers.py 64 256 wgrad > "$out"/layers_r02_64_wgrad9k.txt 2>&1
FDX_WGRAD9_V1=1 timeout 300 python tests/gpu_bench_layers.py 64 256 wgrad > "$out"/layers_r02_64_wgrad9_v1.txt 2>&1
timeout 300 python tests/gpu_bench_layers.py 64 256 gnonly > "$out"/layers_r02_gn_2pass.txt 2>&1
timeout 300 python tests/gpu_bench_layers.py 256 64 gnonly > "$out"/layers_r02_gn256_default.txt 2>&1
timeout 300 python tests/gpu_bench_attention.py > "$out"/layers_r02_attention.txt 2>&1
tail -3 "$out"/layers_r02_64_wgrad9k.txt "$out"/layers_r02_64_wgrad9_v1.txt
tail -2 "$out"/layers_r02_gn_2pass.txt "$out"/layers_r02_gn256_default.txt
cat "$out"/layers_r02_attention.txt
