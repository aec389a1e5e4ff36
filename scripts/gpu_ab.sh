#!/bin/bash
# A/B visit: for every variant "NAME:ENV=VAL,ENV=VAL" run the GPU suite (first variant: whole suite; others: -x) and a short bench.
# usage: gpu_ab.sh TAG "base:" "nopipe:NL_PIPELINE=0" ...
tag=$1; shift; out=gpurun_out/$tag; mkdir -p $out
export NL_BENCH_SKIP_CPU=1
for spec in "$@"; do
  name=${spec%%:*}; envs=${spec#*:}
  (
    IFS=','; for kv in $envs; do [ -n "$kv" ] && export "$kv"; done; unset IFS
    timeout 400 python -m pytest tests -m gpu -q -p no:cacheprovider --timeout 150 -x > $out/pytest_$name.log 2>&1; echo "[$name] pytest rc=$? $(tail -1 $out/pytest_$name.log)"
    timeout 300 python bench.py --steps 10 --warmup 3 > $out/bench_$name.json 2> $out/bench_$name.err; echo "[$name] bench rc=$?"
    python - <<PY
import json
try:
    d=json.load(open("$out/bench_$name.json")); print("[$name]", round(d["value"]/1e6,1), "M/s", round(d["ms_per_step"],4), "ms", {k: (round(v,4) if isinstance(v,float) else "") for k,v in d["stage_ms"].items()}, "frozen", round(d["frozen_decoder"]["ms_per_step"],4), round(d["frozen_decoder"]["mlp_fwd_bwd_ms"],4), "track", round(d["tracking"].get("ms_per_scan",0),2))
except Exception as e: print("[$name] bench parse failed", e)
PY
  )
done
