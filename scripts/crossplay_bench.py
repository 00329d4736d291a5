"""Cost of partnerships (DESIGN.md f14): one cross-play call against the M^2 separate device duplicate matches it replaces,
one roll-out with and without a distinct partner, and one ppo.train iteration with and without a partner.

    python scripts/crossplay_bench.py [--reps 5] [--ms 8 16] [--out profiles/r16_partner_b200.json]

Cross-play: M nets, 100 boards, opponents (c, c); the separate way is make_device_duplicate_evaluate(a, c, key,
team1_partner=b) for every (a, b).  Roll-out: 8192 envs x 32 steps on the CUDA-graph path (one graph per way, captured in
a warm-up call).  ppo.train: ppo.py's shapes (8192 envs x 32 steps, minibatch 1,024, 10 epochs, 10,000 eval envs) for two
iterations, timed as the second iteration's time/* entries (eval, rollout, GAE, update).  The two ways alternate in one
process, each timed with a host clock around work that ends in a device synchronise; the first round is a warm-up and is not
reported.  Medians and ranges are in ms.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import sys
import tempfile
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from brl_b200 import ppo, random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.env import BridgeBidding  # noqa: E402
from brl_b200.evaluation import make_crossplay_evaluate, make_device_duplicate_evaluate  # noqa: E402
from brl_b200.models import init_params, make_forward_pass  # noqa: E402
from brl_b200.roll_out import make_roll_out  # noqa: E402
from scripts.population_bench import _gpu_label  # noqa: E402

DEV = "cuda"
T, N = 32, 8192


def _timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def _alternate(ways, reps):
    """{name: stats of ms} over `reps` alternating rounds after one warm-up round"""
    times = {name: [] for name in ways}
    for r in range(reps + 1):
        for name, fn in ways.items():
            ms = _timed(fn)
            if r:
                times[name].append(ms)
    return {name: dict(median_ms=statistics.median(v), min_ms=min(v), max_ms=max(v), samples=v) for name, v in times.items()}


def bench_crossplay(M, reps, boards=100):
    env = BridgeBidding(table=synthetic_deal_table(100_000, seed=1), device=DEV)
    nets = [init_params(10 + k, DEV) for k in range(M)]
    opp = init_params(99, DEV)
    key = brandom.PRNGKey(0)
    crossplay = make_crossplay_evaluate(env, "relu", "DeepMind", boards)
    dup = make_device_duplicate_evaluate(env, "relu", "DeepMind", boards)
    one = {}

    def batched():
        one["imp"] = crossplay(nets, (opp, opp), key)[1]

    def separate():
        for a in range(M):
            for b in range(M):
                dup(nets[a], opp, key, team1_partner=nets[b])
    out = _alternate({"crossplay": batched, "separate": separate}, reps)
    out["speedup"] = out["separate"]["median_ms"] / out["crossplay"]["median_ms"]
    out["matches"], out["boards"] = M * M, boards
    return out


def bench_rollout(reps):
    env = BridgeBidding(table=synthetic_deal_table(100_000, seed=1), device=DEV)
    config = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode="competitive", num_steps=T,
                  reward_scale=7600.0)
    fp = make_forward_pass("relu", "DeepMind")
    roll_out = make_roll_out(config, env, fp, fp, partner_forward_pass=make_forward_pass("relu", "DeepMind"))
    params, opp, partner = init_params(1, DEV), init_params(2, DEV), init_params(3, DEV)
    state = env.init(env.make_keys(5, N))
    runners = {False: (params, None, state, state.observation, torch.zeros((), dtype=torch.int64, device=DEV), brandom.PRNGKey(1))}
    runners[True] = runners[False]

    def run(partnered):
        def fn():
            runners[partnered] = roll_out(runners[partnered], opp, partner_params=partner if partnered else None)[0]
        return fn
    return _alternate({"plain": run(False), "partnered": run(True)}, reps)


def bench_train(reps, partner_path):
    tables, eval_table = [synthetic_deal_table(100_000, seed=k) for k in range(2)], synthetic_deal_table(100_000, seed=9)
    times = {"plain": [], "partnered": []}
    for r in range(reps + 1):
        for name in times:
            logs = []
            cfg = dict(num_envs=N, num_steps=T, minibatch_size=1024, update_epochs=10, total_timesteps=N * T * 2,
                       save_model=False, lr=1e-6, partner_model_path=partner_path if name == "partnered" else None)
            ppo.train(cfg, brandom.PRNGKey(r), tables=tables, eval_table=eval_table, device=DEV, log_fn=logs.append)
            if r:
                times[name].append({k: v * 1e3 for k, v in logs[-1].items() if k.startswith("time/")})
    out = {}
    for name, v in times.items():
        total = [sum(x.values()) for x in v]
        out[name] = dict(median_ms=statistics.median(total), min_ms=min(total), max_ms=max(total), samples=total,
                         parts_median_ms={k: statistics.median(x[k] for x in v) for k in v[0]})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ms", type=int, nargs="+", default=[8, 16])
    ap.add_argument("--train-reps", type=int, default=2)
    ap.add_argument("--out", default="profiles/r16_partner_b200.json")
    a = ap.parse_args()
    res = dict(gpu=_gpu_label(), reps=a.reps)
    res["crossplay"] = {}
    for M in a.ms:
        res["crossplay"][f"M={M}"] = bench_crossplay(M, a.reps)
        print(f"crossplay M={M}", {k: round(v["median_ms"], 2) for k, v in res["crossplay"][f"M={M}"].items()
                                    if isinstance(v, dict)}, flush=True)
    res["rollout"] = dict(bench_rollout(a.reps), shapes=dict(num_envs=N, num_steps=T))
    print("rollout", {k: round(v["median_ms"], 2) for k, v in res["rollout"].items() if "median_ms" in v}, flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "partner.pkl")
        ppo.save_params(init_params(7, DEV), path)
        res["train_iteration"] = dict(bench_train(a.train_reps, path), shapes=dict(num_envs=N, num_steps=T, minibatch_size=1024,
                                                                                 update_epochs=10, num_eval_envs=10000))
    print("train", {k: round(v["median_ms"], 2) for k, v in res["train_iteration"].items() if "median_ms" in v}, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
