#!/bin/bash
# driver-style bench contract at N = number of visible GPUs (reference arm first), + the two-GPU split test
mkdir -p gpurun_out
cd "$(dirname "$0")/.."
N=$(nvidia-smi -L | wc -l)
run() { # impl
  if [ "$N" = "1" ]; then python bench.py --gpus 1 --steps 20 --warmup 3 "$@"
  else python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29533 bench.py --gpus $N --steps 20 --warmup 3 "$@"; fi
}
echo "== reference arm, N=$N"; ( time run --impl reference ) > gpurun_out/contract_ref_${N}.json 2> gpurun_out/contract_ref_${N}.err; echo "exit $?"; tail -c 600 gpurun_out/contract_ref_${N}.json; grep real gpurun_out/contract_ref_${N}.err
echo "== our arm, N=$N"; ( time run ) > gpurun_out/contract_ours_${N}.json 2> gpurun_out/contract_ours_${N}.err; echo "exit $?"; grep real gpurun_out/contract_ours_${N}.err
python - <<PY
import json
d = json.loads([l for l in open("gpurun_out/contract_ours_${N}.json") if l.startswith("{")][-1])
print({k: d[k] for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "gpu_launches", "timed_region_s")})
print("e2e", d["e2e"]["value"], d["e2e"].get("host_h2d_copy_only_gbs_per_gpu"), "u8", d["e2e_u8_ingest"]["value"], "labels", d["e2e_u8_ingest"]["labels_out"]["value"])
print("clocks", d["clocks"], "parity", d.get("parity_max_rel"), "roofline", d.get("roofline", {}).get("frac"), "cpu", d.get("cpu_baseline", {}).get("value"))
PY
if [ "$N" = "2" ]; then
  echo "== two-GPU split test"; timeout 600 python -m pytest -q --tb=short -p no:cacheprovider -x tests/test_gpu_split2.py -m gpu > gpurun_out/S2.log 2>&1; echo "exit $?"; tail -3 gpurun_out/S2.log
fi
