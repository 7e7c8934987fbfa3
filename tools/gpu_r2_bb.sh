#!/bin/bash
# round 2, call BB: start stagger of the CTAs of the four-pipeline attention kernel (kernel alone, 1 225 tiles) + kernel tests with the
# tail's automatic stagger
mkdir -p gpurun_out
L=gpurun_out/r2bb.log
: > $L
timeout 600 python -m pytest tests/test_gpu_kernels.py tests/test_gpu_fp16.py -m gpu -q --no-header 2>&1 | grep -E "passed|failed|FAILED|Error|error|vitocm:|assert " | head -20 >> $L
for stg in 0 10000 20000 40000 80000 160000 0 40000; do
  echo "attn stagger $stg: $(VITOCM_ATTN_STAGGER=$stg TILES=1225 PRECISION=2 timeout 200 python tools/attn_bench.py 2>&1 | tail -1)" >> $L
done
echo "tail auto stagger: $(VITOCM_MLP_TL_ITEM=20 timeout 200 python tools/tail_timeline.py 1225 2 1 2>&1 | head -1)" >> $L
cat $L
