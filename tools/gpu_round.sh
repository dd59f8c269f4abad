#!/bin/bash
# Helper for gpurun calls: runs the GPU parity tests (and optionally the bench) and leaves logs under gpurun_out/.
#   tools/gpu_round.sh <tag> [bench] [ncu]
tag=${1:-run}; shift
mkdir -p gpurun_out
export PYTHONUNBUFFERED=1
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm --format=csv > gpurun_out/${tag}_smi.txt 2>&1
python - <<'PYEOF' 2>&1 | tee gpurun_out/${tag}_occupancy.txt
import ctypes as C, torch
from nice_slam_b200 import _lib
torch.zeros(1, device="cuda")
a, b = C.c_int(0), C.c_int(0)
print("occupancy rc", _lib.lib().nsb_debug_occupancy(C.byref(a), C.byref(b)), "fwd CTAs/SM", a.value, "bwd CTAs/SM", b.value)
PYEOF
timeout 900 python -m pytest tests -q -m gpu -x 2>&1 | tail -60 > gpurun_out/${tag}_tests.log
echo "pytest exit ${PIPESTATUS[0]}" >> gpurun_out/${tag}_tests.log
tail -15 gpurun_out/${tag}_tests.log
for what in "$@"; do
  case $what in
    bench)
      timeout 900 python bench.py --steps 20 --warmup 5 > gpurun_out/${tag}_bench.json 2> gpurun_out/${tag}_bench.err
      echo "bench exit $?"; tail -c 3000 gpurun_out/${tag}_bench.json; tail -5 gpurun_out/${tag}_bench.err ;;
    simt)
      NSB_MLP_BACKEND=1 timeout 900 python -m pytest tests -q -m gpu 2>&1 | tail -15 > gpurun_out/${tag}_tests_simt.log; tail -3 gpurun_out/${tag}_tests_simt.log ;;
    ncu)
      timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/${tag}_launches.csv python bench.py --steps 2 --warmup 1 > gpurun_out/${tag}_ncu_bench.log 2>&1
      timeout 1200 ncu --set full --clock-control none --import-source on -k regex:render_.*tile -c 4 -o gpurun_out/${tag}_full python bench.py --steps 1 --warmup 1 > gpurun_out/${tag}_ncu_full.log 2>&1
      echo "ncu done" ;;
  esac
done
