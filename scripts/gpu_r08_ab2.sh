# r08 A/B on one B200, second call: bench.py's headline legs alternated between a parent checkout (ab_parent/, built beside
# this tree) and this tree, --sweep once per tree, --dump-outputs from both compared byte for byte, the chained-launch tests.
set -x
O=${OUT:-r08_out}  # results directory
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/r08_card.txt
python -m pytest -q -x -m gpu tests/test_cuda_rollout_chain.py 2>&1 | tail -3 | tee $O/r08_chain_tests.txt
B="--gpus 1 --steps 50 --warmup 5 --no-cpu --no-policy --no-update --no-matches"
for r in 1 2 3; do
  (cd ab_parent && python bench.py $B) 2>/dev/null | tail -1 | sed 's/^/{"tree": "parent", "bench": /; s/$/}/' >> $O/r08_c_bench_ab.jsonl
  python bench.py $B 2>/dev/null | tail -1 | sed 's/^/{"tree": "this change", "bench": /; s/$/}/' >> $O/r08_c_bench_ab.jsonl
done
(cd ab_parent && python bench.py $B --sweep --dump-outputs /tmp/dump_parent) 2>/dev/null | tail -1 | sed 's/^/{"tree": "parent", "bench": /; s/$/}/' >> $O/r08_d_sweep_ab.jsonl
python bench.py $B --sweep --dump-outputs /tmp/dump_change 2>/dev/null | tail -1 | sed 's/^/{"tree": "this change", "bench": /; s/$/}/' >> $O/r08_d_sweep_ab.jsonl
ls -la /tmp/dump_parent /tmp/dump_change
for f in /tmp/dump_parent/*; do cmp "$f" "/tmp/dump_change/$(basename $f)" && echo "identical $(basename $f)"; done | tee $O/r08_e_dump_cmp.txt
rm -rf /tmp/dump_parent /tmp/dump_change
python - "$O" <<'PY'
import json, sys
for l in open(sys.argv[1] + "/r08_c_bench_ab.jsonl"):
    d = json.loads(l); b = d["bench"]
    print(d["tree"], b["value"], b.get("e2e", {}).get("value"))
PY
