#!/bin/bash
# f2b_field_bwd_scatter (field-MLP backward + hash scatter in one kernel): its tests and smoke(), then one bench line per
# configuration of the sweep {4, 8} scatter warps per CTA x {2, 3} CTAs per SM, and one of the two-kernel sequence
cd "$(dirname "$0")/.."
O=${OUT:-/tmp/f2b_r03}; mkdir -p $O; TAG=${TAG:-r03a}   # OUT: where the bench lines and logs go
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/${TAG}_gpu.csv
timeout 900 python -m pytest tests/test_gpu_field_bwd_scatter.py -q -x -p no:cacheprovider 2>&1 | tail -15
timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3
B="python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline --no-ref-gpu"
run() {   # $1 = label, rest = env
  local tag=$1; shift
  env "$@" timeout 600 $B > $O/${TAG}_$tag.json 2> $O/${TAG}_$tag.err; echo "--- $tag rc=$?"
  python - "$O/${TAG}_$tag.json" "$tag" >> $O/${TAG}_sweep.jsonl <<'PY'
import json, sys
d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
k = d["kernels"]
row = {"config": sys.argv[2], "ms_per_step": d["ms_per_step"], "e2e_ms_per_step": d["e2e"]["ms_per_step"],
       "gpu_launches": d["gpu_launches"], "clocks": d["clocks"],
       **{n: k[n]["ms_per_step"] for n in ("f2b_field_bwd_scatter", "f2b_mlp_bwd2", "f2b_hash_bwd") if n in k}}
print(json.dumps(row))
PY
  tail -1 $O/${TAG}_sweep.jsonl
}
run two_kernel F2B_FIELD_BWD_SCATTER=0
for w in 4 8; do for c in 3 2; do run w${w}_c${c} F2B_FIELD_BWD_SCATTER=1 F2B_FBS_WARPS=$w F2B_FBS_CTAS=$c; done; done
run two_kernel_again F2B_FIELD_BWD_SCATTER=0
