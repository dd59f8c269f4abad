#!/bin/bash
# ncu evidence of the round: launch list of the bench command, full-set captures of the dominant kernels (tile kernels,
# weight-gradient kernel).  Numbers printed under ncu are never bench values.
tag=${1:-ev}
mkdir -p gpurun_out
export PYTHONUNBUFFERED=1
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/${tag}_launches.csv python bench.py --steps 2 --warmup 1 > gpurun_out/${tag}_launches_bench.log 2>&1
echo "launch list exit $?"
NSB_BENCH_FAST=1 timeout 900 ncu --set full --clock-control none --import-source on -k regex:render_.*_tile_kernel -s 8 -c 4 -o gpurun_out/${tag}_full_tile python bench.py --steps 6 --warmup 3 > gpurun_out/${tag}_full_tile.log 2>&1
echo "full tile exit $?"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:render_.*tile_kernel -s 9 -c 3 -o gpurun_out/${tag}_full_map python tools/map_launches.py 996 > gpurun_out/${tag}_full_map.log 2>&1
echo "full map exit $?"
ls -la gpurun_out/${tag}_*
