#!/bin/bash
# Same-box A/B of several builds of the library (run under gpurun): for every ab/<name>.so given, the bit-level digest of a
# fixed scenario (scripts/digest_step.py) and the device-resident bench lines of c2 (16 384 envs) and c5 (30 % resets).
#   python -m leibnizgym_b200.build -o ab/new.so; gpurun -- 'bash scripts/ab_bench.sh base new'
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
EXTRA=${AB_EXTRA:-}
for v in "$@"; do
  export LG_LIB_PATH=$PWD/ab/$v.so
  [ -z "$AB_NO_DIGEST" ] && timeout 300 python scripts/digest_step.py 2>&1 | sed "s/^/[$v] /" | tee gpurun_out/digest_$v.txt | cut -c1-400
  for wl in ${AB_WORKLOADS:-c2 c5}; do
    timeout 300 python bench.py --workload $wl --steps 512 --warmup 64 --no-cpu --no-e2e $EXTRA > gpurun_out/ab_${v}_$wl.json 2> gpurun_out/ab_${v}_$wl.err || tail -3 gpurun_out/ab_${v}_$wl.err
    python - <<PY
import json
try:
    d = json.loads(open("gpurun_out/ab_${v}_$wl.json").read().strip().splitlines()[-1])
    r, t = d["roofline"], d["timing"]
    print("[$v] $wl step %.2f us (cold %.2f) post %.2f pre %.2f frac %.3f whole %.3f copy %.2f" % (
        t["us_per_step"], t["cold_start_us_per_step"], r["launch_us"], r["pre_us"], r["frac"], r["whole_step_frac"], r["device_copy_same_bytes_us"]))
except Exception as ex:
    print("[$v] $wl FAILED", ex)
PY
  done
done
