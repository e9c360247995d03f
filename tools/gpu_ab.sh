#!/bin/bash
# A/B of one environment knob on one box, same minute: quick parity subset, then the bench value and the
# in-step kernel times with the knob off / on, alternating.   usage: tools/gpu_ab.sh KNOB [off_value] [on_value]
KNOB=${1:-CBINFER_FUSE_TAIL}; OFF=${2:-0}; ON=${3:-1}
mkdir -p gpurun_out
cd "$(dirname "$0")/.."
PYT="python -m pytest -q --tb=short -p no:cacheprovider --timeout 600 -x"
echo "== parity subset"; timeout 900 $PYT tests/test_gpu_tiles.py tests/test_gpu_modules.py tests/test_gpu_parity_baseline.py tests/test_gpu_ops.py -m gpu -k "${AB_TESTS:-tile or self or candidate or fused or tail or pipeline or scene or parity or baseline or hint or dilate}" > gpurun_out/ab_pytest.log 2>&1; echo "exit $?"; tail -12 gpurun_out/ab_pytest.log
for rep in 1 2; do
  for v in $OFF $ON; do
    env $KNOB=$v timeout 600 python bench.py --steps 400 --warmup 10 --no-extras > gpurun_out/ab_${v}_$rep.json 2> gpurun_out/ab_${v}_$rep.err
    python - <<PY
import json
try:
    d = json.loads(open("gpurun_out/ab_${v}_$rep.json").read().strip().splitlines()[-1])
    print("$KNOB=$v rep $rep: value %.0f frames/s  ms/step %.4f  e2e %.0f  u8 %.0f" % (d["value"], d["ms_per_step"], d["e2e"]["value"], d.get("e2e_u8_ingest", {}).get("value", 0)))
except Exception as e:
    print("bench parse failed", e); print(open("gpurun_out/ab_${v}_$rep.err").read()[-1500:])
PY
  done
done
for v in $OFF $ON; do
  echo "== in-step kernel times, $KNOB=$v"; env $KNOB=$v timeout 300 python tools/instep_timing.py 2>&1 | tail -14
done
