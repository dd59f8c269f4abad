#!/bin/bash
tag=${1:-q}
mkdir -p gpurun_out
export PYTHONUNBUFFERED=1
timeout 900 python -m pytest tests -q -m gpu 2>&1 | tail -8 > gpurun_out/${tag}_tests.log; echo "pytest exit ${PIPESTATUS[0]}" >> gpurun_out/${tag}_tests.log; tail -4 gpurun_out/${tag}_tests.log
for v in "NSB_X=0"; do
  env $v NSB_BENCH_FAST=1 timeout 600 python bench.py --steps 300 --warmup 10 > gpurun_out/${tag}_fast_${v%%=*}.json 2>/dev/null
  python - <<PYEOF
import json
d=json.load(open("gpurun_out/${tag}_fast_${v%%=*}.json"))
print("fast bench [$v]: ms/step", round(d["ms_per_step"],5), "e2e", round(d["e2e"]["ms_per_step"],5), "warm", round(d["extra"]["l2_warm_ms_per_step"],5), "bwd", round(d["roofline"]["launch_ms"],5))
PYEOF
done
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 200 --csv --log-file gpurun_out/${tag}_map_launches.csv python tools/map_launches.py 996 > gpurun_out/${tag}_map_launches.log 2>&1
python - <<PYEOF
import csv
rows=[r for r in csv.reader(open("gpurun_out/${tag}_map_launches.csv")) if len(r)>10]
hdr=rows[0]; ki=hdr.index("Kernel Name"); vi=hdr.index("Metric Value")
seq=[(r[ki].split("(")[0], float(r[vi])) for r in rows[1:]]
idx=[i for i,(k,_) in enumerate(seq) if "render_fwd" in k]
for k,v in seq[idx[-1]:]: print("%-60s %10.1f us" % (k[:60], v/1000 if v>1000 else v))
PYEOF
