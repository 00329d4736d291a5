# r08 A/B on one B200, third call: bench.py's headline legs alternated between the parent checkout (ab_parent/), this
# tree, and this tree with every launch (caller-supplied uniforms too) made with programmatic dependent launch
set -x
O=${OUT:-r08_out}  # results directory
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/r08_card.txt
python -m pytest -q -x -m gpu tests/test_cuda_rollout_chain.py 2>&1 | tail -3 | tee $O/r08_chain_tests.txt
B="--gpus 1 --steps 50 --warmup 5 --no-cpu --no-policy --no-update --no-matches"
for r in 1 2 3; do
  (cd ab_parent && python bench.py $B) 2>/dev/null | tail -1 | sed 's/^/{"tree": "parent", "bench": /; s/$/}/' >> $O/r08_c_bench_ab.jsonl
  python bench.py $B 2>/dev/null | tail -1 | sed 's/^/{"tree": "this change", "bench": /; s/$/}/' >> $O/r08_c_bench_ab.jsonl
  BRL_B200_LIB=brl_b200/lib/libbrl_pdlall.so python bench.py $B 2>/dev/null | tail -1 | sed 's/^/{"tree": "pdl for caller uniforms too", "bench": /; s/$/}/' >> $O/r08_c_bench_ab.jsonl
done
python scripts/exp_launch_fixed_cost.py --label "this change" --out $O/r08_b_fixed_cost.jsonl > /dev/null
python - "$O" <<'PY'
import json, sys
for l in open(sys.argv[1] + "/r08_c_bench_ab.jsonl"):
    d = json.loads(l); b = d["bench"]
    print(d["tree"], b["value"], b.get("e2e", {}).get("value"))
PY
