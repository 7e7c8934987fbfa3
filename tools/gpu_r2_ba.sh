#!/bin/bash
# round 2, call BA: start stagger of the CTA pairs of the folded block tail, wider sweep (kernel alone) + the bench step
mkdir -p gpurun_out
L=gpurun_out/r2ba.log
: > $L
for stg in 0 90000 120000 150000 180000 240000 360000; do
  echo "stagger $stg: $(VITOCM_TAIL_STAGGER=$stg VITOCM_MLP_TL_ITEM=20 timeout 200 python tools/tail_timeline.py 1225 2 1 2>&1 | head -1) | 175 tiles: $(VITOCM_TAIL_STAGGER=$stg VITOCM_MLP_TL_ITEM=4 timeout 200 python tools/tail_timeline.py 175 2 1 2>&1 | head -1 | sed 's/.*: //')" >> $L
done
for rep in 0 1; do
  for stg in 0 120000 180000; do
    VITOCM_TAIL_STAGGER=$stg timeout 300 python bench.py --no-cpu-baseline --no-extras > gpurun_out/r2ba_bench_${stg}_${rep}.json 2> gpurun_out/r2ba_bench_${stg}_${rep}.err
    python - $stg $rep >> $L <<'PY'
import json, sys
b, rep = sys.argv[1:3]
try:
    d = json.loads(open(f"gpurun_out/r2ba_bench_{b}_{rep}.json").read().strip().splitlines()[-1])
    kc = {k: round(v["ms"], 2) for k, v in d["kernel_classes"].items()}
    print("stagger", b, "rep", rep, d["dtype"], round(d["value"], 1), d["unit"], round(d["ms_per_step"], 2), "ms e2e", round(d["e2e"]["value"], 1), kc, d["clocks"]["sm_mhz"])
except Exception as e:
    print("bench ERR", b, rep, repr(e))
PY
  done
done
cat $L
