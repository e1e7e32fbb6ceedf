#!/bin/bash
# k_step_inc with the every-CTA-works grid (2 update rounds per warp from 48 Ki envs) against the three-launch path:
# where should pcgrl_step switch?
set -u
mkdir -p gpurun_out
run() {
  n=$1; path=$2; shift 2
  env PCGRL_STEP_PATH=$path "$@" timeout 200 python bench.py --envs $n --steps 300 --warmup 10 --no-e2e --no-cpu-baseline --no-configs 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('envs=$n path=$path $*', 'value %.4g'%d['value'], 'ms/step %.4f'%d['ms_per_step'], 'kernel_ms %.4f'%d['roofline']['kernel_ms_per_launch'])"
}
{
run 98304 incfused
run 163840 incfused
run 163840 inc
run 262144 incfused
run 262144 inc
run 393216 incfused
run 393216 inc
run 524288 incfused
run 524288 inc
} | tee gpurun_out/step_inc_switch.txt
