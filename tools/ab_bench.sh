#!/bin/bash
# A/B runs of the default bench command under different environment switches (run under gpurun,
# one GPU).  Every argument is one configuration: a space-separated list of VAR=value pairs
# ("A=1" = the defaults).  Prints frames/s and the CUDA-event stage times of each.
#   bash tools/ab_bench.sh "A=1" "DH_BOX_BANDS=1" "DH_TRAV_THREADS=512 DH_GATE_CTAS=2" "A=1"
cd "$(dirname "$0")/.." || exit 1
mkdir -p gpurun_out
for cfg in "$@"; do
  # shellcheck disable=SC2086
  env $cfg python bench.py --steps "${STEPS:-5}" --warmup 3 --no-cpu-baseline 2>/dev/null | tail -1 > gpurun_out/ab_tmp.json
  python - "$cfg" <<'PY'
import json, sys
d = json.loads(open("gpurun_out/ab_tmp.json").read())
st = {k: round(v, 4) for k, v in d["stage_ms_per_step"].items() if v}
print("%-40s %8d frames/s  %s  e2e_biwi %d" % (sys.argv[1], round(d["value"]), st, round(d["e2e_biwi"]["value"])))
PY
done
