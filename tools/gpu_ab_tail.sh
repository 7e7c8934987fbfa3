#!/bin/bash
# A/B of two builds of libvitocm.so on the block tail alone (folded form): tools/bin/libvitocm_a.so (A) against the in-tree build (B).
# (tools/tail_timeline.py runs vitocm_block_tail_folded; the A build must export every symbol of include/vitocm.h, which
# _lib.load_library checks, so it is built from a tree that has vitocm_block_tail_folded.)
#   bash tools/gpu_ab_tail.sh <log name> [test files...]
mkdir -p gpurun_out
L=gpurun_out/$1.log
shift
: > $L
if [ $# -gt 0 ]; then
  timeout 900 python -m pytest "$@" -m gpu -q --no-header 2>&1 | grep -E "passed|failed|FAILED|Error|error|vitocm:|assert " | head -30 >> $L
fi
for rep in 0 1 2; do
  for b in a b; do
    if [ $b = a ]; then export VITOCM_LIB=$PWD/tools/bin/libvitocm_a.so; else unset VITOCM_LIB; fi
    echo "build $b rep $rep: $(VITOCM_MLP_TL_ITEM=20 timeout 200 python tools/tail_timeline.py 1225 2 1 2>&1 | grep -E 'us/launch|OUT complete|next norm1|ep1 steps' | tr '\n' '|')" >> $L
  done
done
cat $L
