#!/bin/bash
OUT=gpurun_out; mkdir -p $OUT
CMD="python bench.py --steps 3 --warmup 3 --skip-e2e --skip-cpu-baseline --rff-split off"
$CMD > $OUT/r2f_plain.log 2>&1 &&
ncu --set full --clock-control none --import-source on --kernel-name-base mangled -k regex:Li2ELi2EE -s 4 -c 1 -o $OUT/r2f_prof_rff $CMD > $OUT/r2f_ncu.log 2>&1; echo "ncu=$?"
