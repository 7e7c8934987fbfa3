#!/bin/bash
# round 2, call AS: block tail, ep 2 statistics pass writes OUT + b2 back to TMEM (build B) against the fold-only build A: tests of B,
# kernel alone (tools/tail_timeline.py, folded form) A/B interleaved
mkdir -p gpurun_out
L=gpurun_out/r2as.log
: > $L
timeout 900 python -m pytest tests/test_gpu_fp16.py tests/test_gpu_kernels.py tests/test_gpu_parity.py -m gpu -q --no-header 2>&1 | grep -E "passed|failed|FAILED|Error|error|vitocm:|assert " | head -30 >> $L
for rep in 0 1 2; do
  for b in a b; do
    if [ $b = a ]; then export VITOCM_LIB=$PWD/tools/bin/libvitocm_a.so; else unset VITOCM_LIB; fi
    echo "build $b rep $rep: $(VITOCM_MLP_TL_ITEM=20 timeout 200 python tools/tail_timeline.py 1225 2 1 2>&1 | head -1)" >> $L
  done
done
cat $L
