"""Cost of the KL anchor at ppo.py's shapes: one roll-out with and without the anchor's forward, and one update step,
anchored and plain, for K = 1 (make_update_step) and K = 4 (make_population_update_step).

    python scripts/anchor_kl_bench.py [--reps 6] [--ks 1 4] [--out profiles/r14_anchor_kl_b200.json]

Shapes: 8192 envs x 32 steps, minibatch 1,024, 10 epochs (2,560 optimizer steps per update).  The roll-out is the
CUDA-graph path of roll_out.make_roll_out (one graph per way, captured in a warm-up call).  Updates run on synthetic
rollouts (sparse 0/1 bf16 observations, random legal masks and actions) with anchor logits that differ from the policy,
anchor_kl_coef = 0.1.  The two ways alternate in one process, each timed with a host clock around work that ends in a
device synchronise; the first pair is a warm-up and is not reported.  Medians and ranges are given in ms.  The card's name
and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from brl_b200 import random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.env import BridgeBidding  # noqa: E402
from brl_b200.models import init_params, make_forward_pass  # noqa: E402
from brl_b200.optim import make_optimizer  # noqa: E402
from brl_b200.roll_out import make_roll_out  # noqa: E402
from brl_b200.update import make_population_update_step, make_update_step  # noqa: E402
from scripts.population_bench import _config, _gpu_label, _rollout  # noqa: E402

DEV = "cuda"
T, N, MBS, EPOCHS = 32, 8192, 1024, 10


def _timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def _alternate(ways, reps):
    """{name: [ms]} over `reps` alternating rounds after one warm-up round"""
    times = {name: [] for name in ways}
    for r in range(reps + 1):
        for name, fn in ways.items():
            ms = _timed(fn)
            if r:
                times[name].append(ms)
    return {name: dict(median_ms=statistics.median(v), min_ms=min(v), max_ms=max(v), samples=v) for name, v in times.items()}


def bench_rollout(reps):
    env = BridgeBidding(table=synthetic_deal_table(100_000, seed=1), device=DEV)
    config = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode="competitive", num_steps=T,
                  reward_scale=7600.0)
    fp = make_forward_pass("relu", "DeepMind")
    roll_out = make_roll_out(config, env, fp, fp, make_forward_pass("relu", "DeepMind"))
    params, opp, anchor = init_params(1, DEV), init_params(2, DEV), init_params(3, DEV)
    state = env.init(env.make_keys(5, N))
    runners = {False: (params, None, state, state.observation, torch.zeros((), dtype=torch.int64, device=DEV), brandom.PRNGKey(1))}
    runners[True] = runners[False]

    def run(anchored):
        def fn():
            runners[anchored] = roll_out(runners[anchored], opp, anchor_params=anchor if anchored else None)[0]
        return fn
    return _alternate({"plain": run(False), "anchored": run(True)}, reps)


def bench_update(K, reps):
    fp = make_forward_pass("relu", "DeepMind", precision="tc")
    configs = [dict(_config(k, T, N, MBS, EPOCHS), anchor_kl_coef=0.1) for k in range(K)]
    rollouts = [_rollout(100 + k, T, N) for k in range(K)]
    g = torch.Generator(device=DEV).manual_seed(7)
    anchors = [torch.randn((T, N, 38), generator=g, device=DEV) for _ in range(K)]
    params = [init_params(k, DEV) for k in range(K)]
    opts = [make_optimizer(c) for c in configs]
    runners = [(p, o.init(p), None, None, 0, brandom.PRNGKey(k)) for k, (p, o) in enumerate(zip(params, opts))]
    if K == 1:
        step = make_update_step(configs[0], fp, opts[0])

        def run(anchored):
            kw = {"anchor_logits": anchors[0]} if anchored else {}
            return lambda: step(runners[0], *rollouts[0], **kw)
    else:
        step = make_population_update_step(configs, fp, opts)

        def run(anchored):
            kw = {"anchor_logits": anchors} if anchored else {}
            return lambda: step(runners, [r[0] for r in rollouts], [r[1] for r in rollouts], [r[2] for r in rollouts], **kw)
    out = _alternate({"plain": run(False), "anchored": run(True)}, reps)
    for way in out.values():
        way["per_optimizer_step_ms"] = way["median_ms"] / (EPOCHS * T * N // MBS)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--ks", type=int, nargs="+", default=[1, 4])
    ap.add_argument("--out", default="profiles/r14_anchor_kl_b200.json")
    a = ap.parse_args()
    res = dict(gpu=_gpu_label(), shapes=dict(num_envs=N, num_steps=T, minibatch_size=MBS, update_epochs=EPOCHS), reps=a.reps)
    res["rollout"] = bench_rollout(a.reps)
    print("rollout", {k: round(v["median_ms"], 2) for k, v in res["rollout"].items()}, flush=True)
    res["update"] = {}
    for K in a.ks:
        res["update"][f"K={K}"] = bench_update(K, a.reps)
        print(f"update K={K}", {k: round(v["median_ms"], 2) for k, v in res["update"][f"K={K}"].items()}, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
