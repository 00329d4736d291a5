# r08 on one B200, final tree: smoke(), the GPU test suite, and bench.py's headline legs with --sweep
set -x
O=${OUT:-r08_out}  # results directory
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2 | tee $O/final_smoke.txt
timeout 420 python -m pytest -q -m gpu tests -p no:cacheprovider 2>&1 | tail -15 | tee $O/final_gpu_tests.txt
python bench.py --gpus 1 --steps 50 --warmup 5 --no-cpu --no-policy --no-update --no-matches --sweep 2>/dev/null | tail -1 > $O/final_bench.json
