#!/bin/bash
# f2b_field_bwd_scatter A/B (TAG=r03c: after the weight-gradient flush every f2b_mlp_bwd2 chain of tiles): the 12 x 2 point of the sweep; five no-flag bench runs per arm, alternating
# (A = F2B_FIELD_BWD_SCATTER=0, the two-kernel sequence; B = the fused kernel); --dump-outputs of A, A again and B;
# a timeline of each arm; the whole GPU suite
cd "$(dirname "$0")/.."
O=${OUT:-/tmp/f2b_r03}; mkdir -p $O; TAG=${TAG:-r03b}   # OUT: where the bench lines and logs go
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/${TAG}_gpu.csv
summ() {   # $1 = bench json, $2 = label, $3 = jsonl
  python - "$1" "$2" >> $3 <<'PY'
import json, sys
d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
k = d["kernels"]
row = {"config": sys.argv[2], "ms_per_step": d["ms_per_step"], "e2e_ms_per_step": d["e2e"]["ms_per_step"],
       "gpu_launches": d["gpu_launches"], "sm_mhz": d["clocks"]["sm_mhz"], "power_w_max": d["clocks"].get("power_w_max"),
       **{n: k[n]["ms_per_step"] for n in ("f2b_field_bwd_scatter", "f2b_mlp_bwd2", "f2b_hash_bwd") if n in k}}
print(json.dumps(row))
PY
  tail -1 $3
}
S="python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline --no-ref-gpu"
for c in "12 2" "8 2"; do set -- $c
  env F2B_FBS_WARPS=$1 F2B_FBS_CTAS=$2 timeout 600 $S > $O/${TAG}_w$1_c$2.json 2>/dev/null; summ $O/${TAG}_w$1_c$2.json w$1_c$2 $O/${TAG}_sweep.jsonl
done
for i in 1 2 3 4 5; do
  F2B_FIELD_BWD_SCATTER=0 timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 > $O/${TAG}_A$i.json 2>$O/${TAG}_A$i.err
  summ $O/${TAG}_A$i.json A$i $O/${TAG}_ab.jsonl
  F2B_FIELD_BWD_SCATTER=1 timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 > $O/${TAG}_B$i.json 2>$O/${TAG}_B$i.err
  summ $O/${TAG}_B$i.json B$i $O/${TAG}_ab.jsonl
done
F2B_FIELD_BWD_SCATTER=0 timeout 600 $S --dump-outputs /tmp/dA > /dev/null 2>&1
F2B_FIELD_BWD_SCATTER=0 timeout 600 $S --dump-outputs /tmp/dA2 > /dev/null 2>&1
F2B_FIELD_BWD_SCATTER=1 timeout 600 $S --dump-outputs /tmp/dB > /dev/null 2>&1
python - > $O/${TAG}_outputs.json <<'PY'
import json, os
import numpy as np
def load(d): return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}
A, A2, B = load("/tmp/dA"), load("/tmp/dA2"), load("/tmp/dB")
rel = lambda a, b: float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b.astype(np.float64)), 1e-300))
out = {}
for k in A:
    out[k] = {"A_vs_B_bit_identical": bool(np.array_equal(A[k].view(np.uint8), B[k].view(np.uint8))),
              "A_vs_A_bit_identical": bool(np.array_equal(A[k].view(np.uint8), A2[k].view(np.uint8))),
              "A_vs_B_rel_l2": rel(B[k], A[k]), "A_vs_A_rel_l2": rel(A2[k], A[k]), "n": int(A[k].size)}
print(json.dumps(out, indent=1))
PY
cat $O/${TAG}_outputs.json
for arm in 0 1; do
  F2B_FIELD_BWD_SCATTER=$arm timeout 600 python scripts/timeline.py > $O/${TAG}_timeline_fbs$arm.json 2>/dev/null
  python - $O/${TAG}_timeline_fbs$arm.json $arm <<'PY'
import json, sys
t = json.load(open(sys.argv[1]))
main = max(t["streams"].items(), key=lambda kv: kv[1]["busy_us"])
names = ("field_bwd_scatter", "mlp_bwd_rc_kernel<0>", "hash_bwd_kernel")
seg = {r["name"]: r["dur_us"] for s in t["streams"].values() for r in s["by_kernel"] if any(n in r["name"] for n in names)}
print(json.dumps({"arm": sys.argv[2], "step_us": t["step_us_under_profiler"], "idle_union_us": t["idle_us"],
                  "main_stream": main[0], "main_busy_us": main[1]["busy_us"],
                  "main_idle_us": round(t["step_us_under_profiler"] - main[1]["busy_us"], 1), "segment_kernels_us": seg}))
PY
done
timeout 900 python -m pytest tests/test_gpu_field_bwd_scatter.py -q -p no:cacheprovider 2>&1 | tail -4
timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -2
timeout 1500 python -m pytest tests -m gpu -q -p no:cacheprovider -rs 2>&1 | tail -25 | tee $O/${TAG}_pytest_gpu.log
