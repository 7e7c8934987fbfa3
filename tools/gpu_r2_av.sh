#!/bin/bash
# round 2, call AV: timeline of one block-tail item (folded form), builds A (two-pass statistics) and B (single sweep)
mkdir -p gpurun_out
L=gpurun_out/r2av.log
: > $L
for b in a b; do
  if [ $b = a ]; then export VITOCM_LIB=$PWD/tools/bin/libvitocm_a.so; else unset VITOCM_LIB; fi
  echo "=== build $b" >> $L
  VITOCM_MLP_TL_ITEM=20 timeout 200 python tools/tail_timeline.py 1225 2 1 >> $L 2>&1
done
cat $L
