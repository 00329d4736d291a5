"""Cost of population-based training (ppo.train_population(..., pbt=...)) at ppo.train's shapes.

    python scripts/pbt_bench.py [--ks 4 8] [--boards 100] [--calls 20] [--iterations 4] [--reps 2]
                                [--out profiles/r13_pbt_b200.json]

For each K it reports:
- ranking: one league fitness call (pbt.league_fitness: a round robin of K nets on `--boards` boards of a 100,000-deal eval
  table in one make_selfplay_league_evaluate call, packing included), median of `--calls` calls after two warm-ups, each
  timed with a host clock around a call that ends in its host read of the statistics;
- iterations: train_population with PBT ranking every iteration (interval 1, the league metric) against the same
  population without PBT (ppo.train's defaults: 8192 envs x 32 steps, minibatch 1,024, 10 epochs, 10,000-env
  evaluations; different seeds, lr and ent_coef), the two alternating `--reps` times.  Each iteration is timed between
  consecutive log callbacks of learner 0; iteration 0 is left out, the medians of the others are reported;
- in the PBT runs, each ranking's fitness call and each exploit step (the device copies of params, mu and nu, the
  config change and the optimizer rebuild), each timed between two device synchronisations the bench adds around it.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from brl_b200 import pbt, ppo  # noqa: E402
from brl_b200 import random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.env import BridgeBidding  # noqa: E402
from brl_b200.evaluation import make_selfplay_league_evaluate  # noqa: E402
from brl_b200.models import init_params  # noqa: E402

DEV = "cuda"


def _gpu_label():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def _med(x):
    return sorted(x)[len(x) // 2] if x else None


def bench_ranking(K, boards, calls):
    env = BridgeBidding(table=synthetic_deal_table(100_000, seed=10_000), device=DEV)
    league = make_selfplay_league_evaluate(env, "relu", "DeepMind", boards)
    nets = [init_params(k, DEV) for k in range(K)]
    key = brandom.PRNGKey(0)
    for _ in range(2):
        pbt.league_fitness(league, nets, key)
    ms = []
    for _ in range(calls):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pbt.league_fitness(league, nets, key)
        ms.append((time.perf_counter() - t0) * 1e3)
    return dict(ranking_ms=ms, ranking_median_ms=_med(ms), matches=K * (K - 1) // 2, boards=boards)


class _Timed(pbt.PopulationBasedTraining):
    """the PBT control plane with its fitness calls and exploit steps timed between device synchronisations"""
    fitness_ms, exploit_ms = [], []

    def fitness(self, learners):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = super().fitness(learners)
        torch.cuda.synchronize()
        _Timed.fitness_ms.append((time.perf_counter() - t0) * 1e3)
        return out

    def exploit(self, loser, winner, factors):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        super().exploit(loser, winner, factors)
        torch.cuda.synchronize()
        _Timed.exploit_ms.append((time.perf_counter() - t0) * 1e3)


def bench_iterations(K, iterations, reps, boards):
    T, n = 32, 8192
    configs = [dict(seed=k, lr=1e-6 * (1 + k), ent_coef=0.001 * (1 + k), save_model=False, total_timesteps=T * n * iterations)
               for k in range(K)]
    tables = [synthetic_deal_table(100_000, seed=k) for k in range(2)]
    eval_table = synthetic_deal_table(100_000, seed=10_000)
    _Timed.fitness_ms, _Timed.exploit_ms = [], []
    pbt.PopulationBasedTraining = _Timed              # what train_population builds
    times = {"plain": [], "pbt": []}
    parents = []
    try:
        for rep in range(reps):
            for name in (("plain", "pbt") if rep % 2 == 0 else ("pbt", "plain")):
                stamps = []
                logs = ppo.train_population(configs, [brandom.PRNGKey(k) for k in range(K)], tables=tables,
                                            eval_table=eval_table, log_fns=[lambda log: stamps.append(time.perf_counter())]
                                            + [None] * (K - 1),
                                            pbt=dict(interval=1, league_boards=boards) if name == "pbt" else None)
                times[name] += [1e3 * (b - a) for a, b in zip(stamps, stamps[1:])]
                if name == "pbt":
                    parents.append([[lg[1][i].get("pbt/parent") for lg in logs] for i in range(1, iterations)])
                del logs
                torch.cuda.empty_cache()
    finally:
        pbt.PopulationBasedTraining = _Timed.__bases__[0]
    plain, with_pbt = _med(times["plain"]), _med(times["pbt"])
    return dict(K=K, iterations_per_run=iterations, plain_iteration_ms=times["plain"], pbt_iteration_ms=times["pbt"],
                plain_median_ms=plain, pbt_median_ms=with_pbt, pbt_overhead_ms=with_pbt - plain,
                in_run_fitness_ms=_Timed.fitness_ms, in_run_fitness_median_ms=_med(_Timed.fitness_ms),
                exploit_ms=_Timed.exploit_ms, exploit_median_ms=_med(_Timed.exploit_ms), parents=parents)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--ks", type=int, nargs="*", default=[4, 8])
    ap.add_argument("--boards", type=int, default=100)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--iterations", type=int, default=4)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out")
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("pbt_bench needs a CUDA device")
    res = dict(device=_gpu_label(), num_envs=8192, num_steps=32, minibatch_size=1024, update_epochs=10, results=[])
    for K in a.ks:
        r = dict(bench_ranking(K, a.boards, a.calls), **bench_iterations(K, a.iterations, a.reps, a.boards))
        print(json.dumps(r), flush=True)
        res["results"].append(r)
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "results"}))


if __name__ == "__main__":
    main()
