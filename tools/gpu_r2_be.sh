#!/bin/bash
# round 2, call BE: timeline of block-tail items with the start stagger (default) and without
mkdir -p gpurun_out
L=gpurun_out/r2be.log
: > $L
for stg in auto 0; do
  for item in 10 30; do
    echo "=== stagger $stg item $item" >> $L
    if [ $stg = auto ]; then unset VITOCM_TAIL_STAGGER; else export VITOCM_TAIL_STAGGER=0; fi
    VITOCM_MLP_TL_ITEM=$item timeout 200 python tools/tail_timeline.py 1225 2 1 >> $L 2>&1
  done
done
cat $L
