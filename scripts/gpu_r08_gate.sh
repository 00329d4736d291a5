# r08 fixed cost per launch on one B200: the t(k) sweep of the rollout kernel and, from a -DBRL_ROLE_TIMING build
# (python scripts/build_variant.py roletiming -DBRL_ROLE_TIMING), its per-phase role clocks
set -x
O=${OUT:-r08_out}  # results directory
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
python scripts/exp_launch_fixed_cost.py --label parent --out $O/r08_a_fixed_cost.jsonl
BRL_B200_LIB=brl_b200/lib/libbrl_roletiming.so python scripts/exp_launch_fixed_cost.py --role --label parent --out $O/r08_a_fixed_cost.jsonl
