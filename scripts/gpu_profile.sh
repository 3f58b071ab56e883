#!/bin/bash
# ncu evidence for profiles/: launch list of the default bench workload (B=4096).  The ncu pass runs only after the same
# command exited 0 without ncu.
mkdir -p gpurun_out
CMD="python bench.py --steps 1 --warmup 3 --no-e2e --no-cpu-baseline --no-serial-leg"
$CMD > gpurun_out/prof_plain.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -c 2000 --csv --log-file gpurun_out/launches.csv $CMD > gpurun_out/ncu_launches.log 2>&1
echo "launch list exit $?"
ls -la gpurun_out | tail -8
