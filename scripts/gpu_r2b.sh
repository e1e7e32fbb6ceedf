#!/bin/bash
# round-2 GPU call B: split / incremental step paths -- parity, then timing of the three paths and the inc knobs
set -u
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_gpu_split.py -x -q 2>&1 | tail -15 | tee gpurun_out/r02b_pytest_split.txt
timeout 900 python -m pytest tests -m gpu -x -q --deselect tests/test_gpu_split.py 2>&1 | tail -6 | tee gpurun_out/r02b_pytest_gpu.txt
for path in fused split inc; do
  echo -n "path=$path: "
  PCGRL_STEP_PATH=$path timeout 200 python bench.py --steps 800 --warmup 10 --no-cpu-baseline --no-configs 2>>gpurun_out/r02b.err | tee gpurun_out/r02b_bench_$path.json | python -c "import json,sys; d=json.loads(sys.stdin.read()); print('value %.4g e2e %.4g kernel_ms %.4f frac %.3f launches %d' % (d['value'], d['e2e']['value'], d['roofline']['kernel_ms_per_launch'], d['roofline']['frac'], d['gpu_launches']))"
done | tee gpurun_out/r02b_paths.txt
for path in fused split inc; do
  echo -n "65k path=$path: "
  PCGRL_STEP_PATH=$path timeout 200 python bench.py --steps 800 --warmup 10 --no-cpu-baseline --no-configs --envs 65536 2>>gpurun_out/r02b.err | python -c "import json,sys; d=json.loads(sys.stdin.read()); print('value %.4g e2e %.4g kernel_ms %.4f' % (d['value'], d['e2e']['value'], d['roofline']['kernel_ms_per_launch']))"
done | tee -a gpurun_out/r02b_paths.txt
tail -5 gpurun_out/r02b.err
