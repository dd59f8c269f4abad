#!/bin/bash
# end-of-round validation on one GPU: smoke(), the GPU suite (default, FP32-FMA back-end, fwd_f16 on), the full bench line
tag=${1:-final}
mkdir -p gpurun_out
export PYTHONUNBUFFERED=1
timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -2
timeout 900 python -m pytest tests -q -m gpu 2>&1 | tail -40 > gpurun_out/${tag}_tests.log; echo "pytest exit ${PIPESTATUS[0]}" >> gpurun_out/${tag}_tests.log; tail -4 gpurun_out/${tag}_tests.log
for v in "NSB_MLP_BACKEND=1" "NSB_FWD_F16=1"; do
  env $v timeout 900 python -m pytest tests -q -m gpu 2>&1 | tail -40 > gpurun_out/${tag}_tests_${v%%=*}_${v#*=}.log; echo "pytest exit ${PIPESTATUS[0]}" >> gpurun_out/${tag}_tests_${v%%=*}_${v#*=}.log
  echo "[$v]"; tail -3 gpurun_out/${tag}_tests_${v%%=*}_${v#*=}.log
done
timeout 1200 python bench.py --steps 300 --warmup 10 > gpurun_out/${tag}_bench.json 2> gpurun_out/${tag}_bench.err
echo "bench exit $?"; python - <<PYEOF
import json
d=json.load(open("gpurun_out/${tag}_bench.json"))
print("ms/step", d["ms_per_step"], "rays/s", d["value"], "e2e", d["e2e"]["ms_per_step"], "warm", d["extra"]["l2_warm_ms_per_step"], "f16", d["extra"]["fwd_f16_option"])
for k in ("mapping_configs1","mapping_loop_step","mapping_loop_step_coarse_mapper"): print(k, d["extra"][k]["ms_per_step"])
print([(x["scene"], round(x["ms_per_step"],3)) for x in d["extra"]["mapping_other_scenes"]])
print("sharded map", d["extra"]["mapping_sharded_masked"]["ms_per_step"])
print([ (x["rays"], x["samples"], round(x["ms_per_step"],3), round(x["rays_per_s"]/1e6,2)) for x in d["extra"]["sweep_tracking_iteration"]])
print("cpu", d["cpu_baseline"])
PYEOF
tail -3 gpurun_out/${tag}_bench.err
