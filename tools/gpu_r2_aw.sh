#!/bin/bash
# round 2, call AW: timeline of block-tail items with the xn_ready stamps (folded form), three different items
mkdir -p gpurun_out
L=gpurun_out/r2aw.log
: > $L
for item in 5 20 35; do
  echo "=== item $item" >> $L
  VITOCM_MLP_TL_ITEM=$item timeout 200 python tools/tail_timeline.py 1225 2 1 >> $L 2>&1
done
cat $L
