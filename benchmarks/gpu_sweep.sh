#!/bin/bash
# development helper: GPU tests, then bench lines for a list of option sets ("defer_pm=500" "defer_pm=800 fused_long=0" ...)
tag=$1; shift
python -m pytest tests -m gpu -x -q > gpurun_out/pytest_$tag.log 2>&1; echo pytest_rc=$?
tail -5 gpurun_out/pytest_$tag.log
i=0
for opts in "$@"; do
  args=""
  for o in $opts; do args="$args --opt $o"; done
  python bench.py --steps 5 --warmup 3 --no-cpu-baseline --no-secondary $args > gpurun_out/bench_${tag}_$i.json 2> gpurun_out/bench_${tag}_$i.err
  echo "== $opts rc=$?"
  python - <<PY
import json
d=json.loads(open("gpurun_out/bench_${tag}_$i.json").read())
r=d["roofline"]
print("qps %.0f e2e %.0f ms/step %.2f kernel_ms %.2f share %.3f launches %d path %s" % (d["value"], d["e2e"]["value"], d["ms_per_step"], r["kernel_ms_per_launch"]*r["launches_per_step"], r["kernel_share_of_step"], r["launches_per_step"], r["path"]))
PY
  i=$((i+1))
done
