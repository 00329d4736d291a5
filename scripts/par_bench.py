"""Cost of the double-dummy par (DESIGN.md f13): the brl_par kernel alone, one roll-out in "score" and in "par_imp" reward
mode, and one ppo.train iteration with and without log_par.

    python scripts/par_bench.py [--reps 6] [--out profiles/r15_par_b200.json]

- brl_par: CUDA events around 200 back-to-back launches at 8,192 and 1,048,576 envs (states from env.init on a
  100,000-row synthetic table, whose 4.8 MB stay in L2), after 20 warm-up launches.
- roll-out: 8192 envs x 32 steps on the CUDA-graph path of roll_out.make_roll_out, one graph per mode captured in a warm-up
  call; the two modes alternate in one process.
- ppo.train: ppo.py's shapes (8192 x 32, minibatch 1,024, 10 epochs, 10,000 eval envs) with the eval/* duplicate match
  played every iteration (num_eval_step = 1), so that every timed iteration pays log_par's extra work; runs of 3
  iterations alternate between log_par False and True, and an iteration's time is the host clock between two successive
  log_fn calls (the first iteration of a run, which captures graphs, is not counted).
Roll-outs and iterations are timed with a host clock around work that ends in a device synchronise.  Medians and ranges
are in ms.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from brl_b200 import ops, ppo  # noqa: E402
from brl_b200 import random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.env import BridgeBidding  # noqa: E402
from brl_b200.models import init_params, make_forward_pass  # noqa: E402
from brl_b200.roll_out import make_roll_out  # noqa: E402
from scripts.anchor_kl_bench import _alternate  # noqa: E402
from scripts.population_bench import _gpu_label  # noqa: E402

DEV = "cuda"
T, N = 32, 8192


def _summary(v):
    return dict(median_ms=statistics.median(v), min_ms=min(v), max_ms=max(v), samples=v)


def bench_par_kernel(n, launches=200):
    env = BridgeBidding(table=synthetic_deal_table(100_000, seed=1), device=DEV)
    state = env.init(env.make_keys(3, n))
    par = torch.empty((n, 4), dtype=torch.float32, device=DEV)
    contract = torch.empty(n, dtype=torch.int32, device=DEV)
    for _ in range(20):
        ops.par(state._packed, env.table, par, contract)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(launches):
        ops.par(state._packed, env.table, par, contract)
    stop.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(stop) / launches
    return dict(n_envs=n, launches=launches, ms_per_launch=ms, envs_per_s=n / ms * 1e3)


def bench_rollout(reps):
    env = BridgeBidding(table=synthetic_deal_table(100_000, seed=1), device=DEV)
    base = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode="competitive", num_steps=T,
                reward_scale=7600.0)
    fp = make_forward_pass("relu", "DeepMind")
    roll_outs = {m: make_roll_out(dict(base, reward_mode=m), env, fp, fp) for m in ("score", "par_imp")}
    params, opp = init_params(1, DEV), init_params(2, DEV)
    state = env.init(env.make_keys(5, N))
    start = (params, None, state, state.observation, torch.zeros((), dtype=torch.int64, device=DEV), brandom.PRNGKey(1))
    runners = {m: start for m in roll_outs}

    def run(m):
        def fn():
            runners[m] = roll_outs[m](runners[m], opp)[0]
        return fn
    return _alternate({m: run(m) for m in roll_outs}, reps)


def bench_train(reps, iterations=3):
    tables, eval_table = [synthetic_deal_table(100_000, seed=k) for k in range(2)], synthetic_deal_table(100_000, seed=9)
    times = {False: [], True: []}
    for r in range(reps):
        for log_par in (False, True):
            stamps = []
            cfg = dict(num_envs=N, num_steps=T, minibatch_size=1024, update_epochs=10, total_timesteps=N * T * iterations,
                       num_eval_envs=10_000, num_eval_step=1, save_model=False, log_par=log_par, log_path="/tmp/par_bench",
                       exp_name=f"r{r}{int(log_par)}")
            ppo.train(cfg, brandom.PRNGKey(r), tables=tables, eval_table=eval_table, device=DEV,
                      log_fn=lambda log: stamps.append(time.perf_counter()))
            times[log_par] += [(b - a) * 1e3 for a, b in zip(stamps[:-1], stamps[1:])]
    return {"log_par=False": _summary(times[False]), "log_par=True": _summary(times[True])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--train-reps", type=int, default=3)
    ap.add_argument("--out", default="profiles/r15_par_b200.json")
    a = ap.parse_args()
    res = dict(gpu=_gpu_label(), shapes=dict(num_envs=N, num_steps=T), reps=a.reps)
    res["brl_par"] = [bench_par_kernel(n) for n in (8192, 1 << 20)]
    print("brl_par", [(r["n_envs"], round(r["ms_per_launch"], 4)) for r in res["brl_par"]], flush=True)
    res["rollout"] = bench_rollout(a.reps)
    print("rollout", {k: round(v["median_ms"], 2) for k, v in res["rollout"].items()}, flush=True)
    res["train_iteration"] = bench_train(a.train_reps)
    print("train iteration", {k: round(v["median_ms"], 1) for k, v in res["train_iteration"].items()}, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
