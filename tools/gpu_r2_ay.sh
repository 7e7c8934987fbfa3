#!/bin/bash
# round 2, call AY: fine stamps of the block tail's ep 2 statistics pass (VITOCM_TAIL_DEBUG=64)
mkdir -p gpurun_out
L=gpurun_out/r2ay.log
: > $L
export VITOCM_TAIL_DEBUG=64
for item in 5 20 35; do
  echo "=== item $item" >> $L
  VITOCM_MLP_TL_ITEM=$item timeout 200 python tools/tail_timeline.py 1225 2 1 2>&1 | grep -E "us/launch|OUT complete|statistics pass|next norm1" >> $L
done
cat $L
