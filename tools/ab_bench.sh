#!/usr/bin/env bash
# Same-box A/B of library builds: tools/ab_bench.sh name=path.so ... ; prints images/s (device-resident, e2e) per build.
# Builds are run round-robin twice so that clock / thermal drift shows up as disagreement between the two passes.
set -u
cd "$(dirname "$0")/.."
for pass in 1 2; do
  for spec in "$@"; do
    name="${spec%%=*}"; rest="${spec#*=}"; path="${rest%%,*}"; envs=""
    [ "${rest}" != "${path}" ] && envs="${rest#*,}"
    env ${envs//,/ } CDC_LIB_PATH="${path}" python bench.py --steps 10 --warmup 3 --no-cpu > "gpurun_out/ab_${name}_${pass}.json" 2>/dev/null
    python - "$name" "$pass" <<'PY'
import json, sys
n, p = sys.argv[1], sys.argv[2]
try:
    d = json.load(open(f"gpurun_out/ab_{n}_{p}.json"))
    print(f"{n:12s} pass {p}: {d['value']:.3f} img/s  e2e {d['e2e']['value']:.3f}  graph {d['roofline'].get('graph_ms', 0):.3f} ms")
except Exception as e:
    print(n, p, "failed", e)
PY
  done
done
