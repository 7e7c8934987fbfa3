#!/bin/bash
# round 2, call AZ: start stagger of the CTA pairs of the folded block tail (kernel alone, 1 225 tiles)
mkdir -p gpurun_out
L=gpurun_out/r2az.log
: > $L
for rep in 0 1; do
  for stg in 0 30000 60000 120000; do
    echo "stagger $stg rep $rep: $(VITOCM_TAIL_STAGGER=$stg VITOCM_MLP_TL_ITEM=20 timeout 200 python tools/tail_timeline.py 1225 2 1 2>&1 | head -1)" >> $L
  done
done
cat $L
