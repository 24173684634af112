#!/bin/bash
# run-to-run spread of the C2 line: the default configuration twice on one box
for v in "FDX_X=0" "FDX_X=1"; do
  echo "== bench c2 $v"
  env $v timeout -s KILL 200 python bench.py --workload c2 --no-cpu-baseline --no-sample --steps 20 2>/dev/null | python -c "
import sys,json
d=json.loads(sys.stdin.read().strip().split('\n')[-1]); print(round(d['value'],1), round(d['ms_per_step'],3), d['clocks']['sm_mhz'])"
done
