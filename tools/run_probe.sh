#!/bin/bash
# Runs every umma_probe case/variant in its own process (a trap in one cannot poison the rest).
mkdir -p gpurun_out
LOG=gpurun_out/probe.log
: > $LOG
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv >> $LOG 2>&1
read NC NP < <(./build/umma_probe count)
VARIANTS=${VARIANTS:-"3 4 5"}
for c in $(seq 0 $((NC-1))); do
  for v in $VARIANTS; do
    timeout 60 ./build/umma_probe $c $v >> $LOG 2>&1
    echo "exit $? (case $c variant $v)" >> $LOG
  done
done
# perf: <idx> <version> <epilogue 0 cast | 1 bias+snake | 2 +residual+raw>
# version: 2 = automatic tiling, 3 = the table's MT/NT, 4 = operand swap disabled
for spec in ${PERF_SPECS:-"0 2 1" "0 4 1" "0 2 0" "1 2 2" "1 4 2" "2 2 1" "2 4 1" "2 3 1" "4 2 1" "5 2 1" "6 2 1" "7 2 2" "7 4 2"}; do
  timeout 120 ./build/umma_probe perf $spec >> $LOG 2>&1
  echo "exit $? (perf $spec)" >> $LOG
done
grep -E "RESULT|PERF|exit [1-9]|prepare failed|timeout|rror" $LOG | cut -c1-170 | tail -100
