#!/bin/bash
# usage: tools/ncu_bench.sh <tag> [kernel-regex]
# Launch list (per-launch gpu time) of a short bench.py run + one --set full capture of the top kernel.
TAG=${1:-r1}; KREGEX=${2:-hh_qr32_c8_kernel}
CMD="python bench.py --steps 3 --warmup 3 --no-cpu --no-extras --e2e-steps 1"
mkdir -p gpurun_out
$CMD > gpurun_out/${TAG}_plain.log 2>&1 || { echo "plain run failed"; tail gpurun_out/${TAG}_plain.log; exit 1; }
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/${TAG}_launches.csv $CMD > gpurun_out/${TAG}_ncu_launches.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:${KREGEX} -s 3 -c 1 -f -o gpurun_out/${TAG}_top $CMD > gpurun_out/${TAG}_ncu_full.log 2>&1
ls -la gpurun_out | tail -8
