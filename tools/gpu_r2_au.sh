#!/bin/bash
# round 2, call AU: block tail, single-sweep statistics with the exact fallback (build B) against the two-pass statistics (build A):
# kernel / fp16 / parity tests of B, kernel alone A/B interleaved, bench step A/B
mkdir -p gpurun_out
L=gpurun_out/r2au.log
: > $L
timeout 900 python -m pytest tests/test_gpu_kernels.py tests/test_gpu_fp16.py tests/test_gpu_parity.py -m gpu -q --no-header 2>&1 | grep -E "passed|failed|FAILED|Error|error|vitocm:|assert " | head -30 >> $L
for rep in 0 1 2; do
  for b in a b; do
    if [ $b = a ]; then export VITOCM_LIB=$PWD/tools/bin/libvitocm_a.so; else unset VITOCM_LIB; fi
    echo "build $b rep $rep: $(VITOCM_MLP_TL_ITEM=20 timeout 200 python tools/tail_timeline.py 1225 2 1 2>&1 | head -1)" >> $L
  done
done
for rep in 0 1; do
  for b in a b; do
    if [ $b = a ]; then export VITOCM_LIB=$PWD/tools/bin/libvitocm_a.so; else unset VITOCM_LIB; fi
    timeout 300 python bench.py --no-cpu-baseline --no-extras > gpurun_out/r2au_bench_${b}_${rep}.json 2> gpurun_out/r2au_bench_${b}_${rep}.err
    python - $b $rep >> $L <<'PY'
import json, sys
b, rep = sys.argv[1:3]
try:
    d = json.loads(open(f"gpurun_out/r2au_bench_{b}_{rep}.json").read().strip().splitlines()[-1])
    kc = {k: round(v["ms"], 2) for k, v in d["kernel_classes"].items()}
    print("build", b, "rep", rep, d["dtype"], round(d["value"], 1), d["unit"], round(d["ms_per_step"], 2), "ms e2e", round(d["e2e"]["value"], 1), kc, d["clocks"]["sm_mhz"])
except Exception as e:
    print("bench ERR", b, rep, repr(e))
PY
  done
done
cat $L
