"""Host loop against device loop for the three evaluations of every ppo.train iteration, at ppo.train's default shapes.

    python scripts/device_eval_bench.py [--reps 10] [--warmup 2] [--out profiles/r05_device_eval_b200.json]

Shapes: train/score -- make_simple_evaluate (host loop: quad steps, both nets forwarded over all 10,000 envs every step)
against make_device_simple_evaluate; eval/* -- make_evaluate(duplicate=True) (host loop: one host read of the two team counts
per step) against make_device_evaluate(duplicate=True), 10,000 envs, in the competitive and the free-run game mode; and the
imp_opp / PFSP probe -- make_simple_duplicate_evaluate against make_device_duplicate_evaluate on 100 boards.  Each timed call
is a whole evaluation, from the keys to its result on the host, between CUDA events; the two loops alternate call by call after
`warmup` calls of each, and every timed pair must give bit-equal per-env returns (R, or cum_return).  The card's name and
power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, ops, random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.evaluation import (make_device_duplicate_evaluate, make_device_evaluate,  # noqa: E402
                                 make_device_simple_evaluate, make_evaluate, make_simple_duplicate_evaluate,
                                 make_simple_evaluate)
from brl_b200.models import LAYERS, init_params  # noqa: E402


def seeded_params(seed, dev):
    p = init_params(seed, dev)   # haiku init with the policy head scaled so that logits have a trained net's magnitude
    p[LAYERS[4]]["w"] *= 128
    return p


def timed(fn):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    out = fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end), out


def compare(name, host_fn, dev_fn, reps, warmup):
    """host_fn / dev_fn return (result, per-env returns); the returns must be bit-equal"""
    for _ in range(warmup):
        host_fn()
        dev_fn()
    t_host, t_dev = [], []
    for _ in range(reps):
        th, (_, rh) = timed(host_fn)
        td, (_, rd) = timed(dev_fn)
        if not torch.equal(rh, rd):
            raise SystemExit(f"{name}: device loop and host loop per-env returns differ")
        t_host.append(th)
        t_dev.append(td)
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    row = {"shape": name, "host_ms": t_host, "device_ms": t_dev, "host_median_ms": med(t_host), "device_median_ms": med(t_dev),
           "speedup": med(t_host) / med(t_dev), "bit_equal_returns": True}
    print(json.dumps({k: v for k, v in row.items() if not k.endswith("_ms") or "median" in k}))
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="profiles/r05_device_eval_b200.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    env = BridgeBidding(table=synthetic_deal_table(10_000, seed=1), device=dev)
    key = brandom.PRNGKey(0)
    actor, opp = seeded_params(900, dev), seeded_params(901, dev)
    n = 10_000   # ppo.train's num_eval_envs
    rows = []

    trace = []
    host_s = make_simple_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, team2_params=opp)
    dev_s = make_device_simple_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, team2_params=opp)

    def host_simple():
        trace.clear()
        r = host_s(actor, key, trace=trace)
        return float(r), trace[-1][1]

    rows.append(compare(f"simple_evaluate_{n}", host_simple, lambda: (float(dev_s(actor, key)), dev_s.buffers.cum_return),
                        args.reps, args.warmup))

    for game_mode in ("competitive", "free-run"):
        seen = {}
        orig = ops.eval_summary

        def spy(acc, cum_return, *a, **kw):
            seen["cum_return"] = cum_return
            return orig(acc, cum_return, *a, **kw)

        cfg = (env, "relu", "DeepMind", "relu", "DeepMind", None, n, game_mode)
        host_e = make_evaluate(*cfg, duplicate=True, team2_params=opp)
        dev_e = make_device_evaluate(*cfg, duplicate=True, team2_params=opp)

        def host_full():
            ops.eval_summary = spy
            try:
                log = host_e(actor, key)[0]
            finally:
                ops.eval_summary = orig
            return log, seen["cum_return"]

        rows.append(compare(f"duplicate_evaluate_{game_mode}_{n}", host_full,
                            lambda: (dev_e(actor, key)[0], dev_e.buffers.cum_return), args.reps, args.warmup))

    probe = 100   # ppo.train's num_prioritized_envs: imp_opp, imp_opp_before / after and the PFSP probe over the zoo
    host_p = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", probe)
    dev_p = make_device_duplicate_evaluate(env, "relu", "DeepMind", probe)
    rows.append(compare(f"duplicate_probe_{probe}", lambda: (lambda r: (r[0], r[3]))(host_p(actor, opp, key)),
                        lambda: (lambda r: (r[0], r[3]))(dev_p(actor, opp, key)), args.reps, args.warmup))
    result = {"card": card, "reps": args.reps, "warmup": args.warmup,
              "timing": "CUDA events around whole evaluations (keys to host result), loops alternating", "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"card": card, "out": args.out}))


if __name__ == "__main__":
    main()
