#!/bin/bash
# ncu --set full capture of the block-aggregation kernels on a 200-cluster batch
TAG=${1:-blk}
ncu --set full --clock-control none --import-source on \
  -k regex:"kA_block_aggregate|kB1_local|kB1_insert|kB3_cluster_emit|k4_probe|k4_commit" -s ${2:-27} -c ${3:-10} \
  -o gpurun_out/prof_${TAG} -f \
  python bench.py --clusters 200 --steps 1 --warmup 3 --no-cpu-baseline --no-e2e --no-extra > gpurun_out/ncu_${TAG}.log 2>&1
ncu -i gpurun_out/prof_${TAG}.ncu-rep --page raw --csv > gpurun_out/raw_${TAG}.csv 2>/dev/null
ncu -i gpurun_out/prof_${TAG}.ncu-rep --page source --csv --kernel-name regex:kA_block > gpurun_out/src_${TAG}_kA.csv 2>/dev/null
ncu -i gpurun_out/prof_${TAG}.ncu-rep --page source --csv --kernel-name regex:kB3_emit > gpurun_out/src_${TAG}_kB.csv 2>/dev/null
tail -2 gpurun_out/ncu_${TAG}.log | cut -c1-300
