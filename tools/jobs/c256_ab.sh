#!/bin/bash
cd "$(dirname "$0")/../.."
mkdir -p gpurun_out
run() { name=$1; shift
  env "$@" timeout 600 python bench.py --config celeba256 --steps 8 --warmup 3 --no-eager --no-cpu --no-c256 > gpurun_out/r2_c256_$name.json 2> gpurun_out/r2_c256_$name.err
  python - <<PY
import json
try:
    d = json.loads(open("gpurun_out/r2_c256_$name.json").read().strip().splitlines()[-1])
    print("$name", round(d["value"], 1), round(d["ms_per_step"], 2), d["clocks"], round(d["host_enqueue_ms_per_step"], 2))
except Exception as e:
    print("$name failed", e)
PY
}
run base A=1
run nooverlap DDPM_B200_WGRAD_OVERLAP=0
run base2 A=1
