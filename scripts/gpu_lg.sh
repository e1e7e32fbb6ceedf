#!/bin/bash
# GPU-box run for the lane-group step (step_lanegroup.cu): parity of every step path, then ms per step by shard size
# against the one-launch / three-launch thread-per-grid paths.
set -u
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_gpu_split.py -m gpu -x -q -k chunked_host_pipeline 2>&1 | tail -8
sweep() {
  n=$1; path=$2; shift 2
  env PCGRL_STEP_PATH=$path "$@" timeout 200 python bench.py --envs $n --steps 300 --warmup 10 --no-e2e --no-cpu-baseline --no-configs > gpurun_out/lg_tmp.json 2> gpurun_out/lg_tmp.err
  python - "$n" "$path" "$*" <<'PY'
import json, sys
try:
    l = json.loads(open("gpurun_out/lg_tmp.json").read().strip().splitlines()[-1])
    print("envs=%s path=%s %s: value %.4g ms_per_step %.4f kernel_ms %.4f" % (sys.argv[1], sys.argv[2], sys.argv[3], l["value"], l["ms_per_step"], l["roofline"]["kernel_ms_per_launch"]))
except Exception as exc:
    print("envs=%s path=%s FAILED %s" % (sys.argv[1], sys.argv[2], exc)); print(open("gpurun_out/lg_tmp.err").read()[-600:])
PY
}
{
sweep 4096 incfused
sweep 4096 lg
sweep 16384 incfused
sweep 16384 lg
sweep 65536 incfused
sweep 65536 lg
} | tee gpurun_out/lg_paths_by_size.txt
for path in incfused lg; do
  for n in 4096 65536; do
    PCGRL_STEP_PATH=$path timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:k_step -s 20 -c 30 --csv --log-file gpurun_out/lg_ncu_${path}_$n.csv \
      python bench.py --envs $n --steps 40 --warmup 5 --no-e2e --no-cpu-baseline --no-configs > /dev/null 2>&1
    python - "$path" "$n" <<'PY'
import csv, sys
path, n = sys.argv[1], sys.argv[2]
rows = [r for r in csv.reader(open(f"gpurun_out/lg_ncu_{path}_{n}.csv")) if len(r) > 5]
hdr = rows[0]; ki, vi = hdr.index("Kernel Name"), hdr.index("Metric Value")
v = [float(r[vi].replace(",", "")) for r in rows[1:] if r[vi].replace(",", "").replace(".", "").isdigit()]
print("ncu", path, n, rows[1][ki][:40], "n=%d avg_us=%.1f min_us=%.1f" % (len(v), sum(v) / len(v) / 1e3, min(v) / 1e3))
PY
  done
done | tee gpurun_out/lg_ncu_times.txt
