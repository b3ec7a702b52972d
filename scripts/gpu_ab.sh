#!/bin/bash
# A/B of other builds of the library (libsffg_<tag>.so next to the default library, e.g. built from another commit)
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
for v in "" "$@"; do
  if [ -z "$v" ]; then unset SFFG_LIB; else export SFFG_LIB=$PWD/space_filling_forest_star_b200/libsffg_$v.so; fi
  timeout 600 python bench.py --steps 8 --warmup 3 --no-cpu --no-extra > gpurun_out/bench_${v:-default}.log 2>&1
  python - <<PY
import json
try:
    d = json.loads(open("gpurun_out/bench_${v:-default}.log").read().strip().splitlines()[-1])
    print("${v:-default}: value %.4g e2e %.4g kernel_ms %.3f" % (d["value"], d["e2e"]["value"], d["roofline"]["kernel_ms"]))
except Exception as e:
    print("${v:-default} failed", e); print(open("gpurun_out/bench_${v:-default}.log").read()[-1500:])
PY
done
