#!/bin/bash
# usage: tools/ncu_batched.sh <tag> [mgs] [out-dir]   (needs a GPU and Nsight Compute)
set -u
TAG=$1; MGS=${2:-0}; OUT=${3:-ncu_out}
mkdir -p $OUT
python tools/prof_batched.py 16 $MGS > $OUT/${TAG}_plain.log 2>&1 || { echo plain run failed; tail $OUT/${TAG}_plain.log; exit 1; }
# one launch per kernel under the profiler
PROF_REPS=1 ncu --set full --clock-control none --import-source on -k regex:qr32 -o /tmp/${TAG} python tools/prof_batched.py 16 $MGS > $OUT/${TAG}_ncu.log 2>&1
ncu -i /tmp/${TAG}.ncu-rep --page raw --csv > $OUT/${TAG}_raw.csv 2>/dev/null
ncu -i /tmp/${TAG}.ncu-rep --page details --csv > $OUT/${TAG}_details.csv 2>/dev/null
ncu -i /tmp/${TAG}.ncu-rep --page source --csv --print-source sass > $OUT/${TAG}_source.csv 2>/dev/null
ls -la /tmp/${TAG}.ncu-rep $OUT/
SZ=$(stat -c %s /tmp/${TAG}.ncu-rep)
if [ "$SZ" -lt 40000000 ]; then cp /tmp/${TAG}.ncu-rep $OUT/; fi
gzip -f $OUT/${TAG}_source.csv
tail -3 $OUT/${TAG}_plain.log
