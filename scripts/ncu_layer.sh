#!/bin/bash
# ncu evidence for the layer kernel on full C3 (1 GPU): the launch list of one pass and one --set full
# capture (launch 6 = layer 5), which includes the layer's DRAM bytes.
# Each profiler run follows a plain run that exited 0.  gpurun -- 'bash scripts/ncu_layer.sh'
set -u
mkdir -p gpurun_out
CMD="python bench.py --steps 1 --warmup 3 --cpu-seconds 0 --e2e-steps 0"
timeout 120 $CMD > gpurun_out/plain.log 2>&1 || { echo "plain run failed"; tail -5 gpurun_out/plain.log; exit 1; }
echo "== launch list"
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 200 --csv --log-file gpurun_out/launches.csv $CMD > gpurun_out/ncu1.log 2>&1; echo "exit $?"
echo "== full capture"
timeout 600 ncu --set full --clock-control none --import-source on -k regex:layer_kernel -s 5 -c 1 -f -o gpurun_out/prof_layer $CMD > gpurun_out/ncu2.log 2>&1; echo "exit $?"
