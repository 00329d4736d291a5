"""Host loop against device loop for whole duplicate matches, on the same seeded nets and keys.

    python scripts/duplicate_match_bench.py [--reps 10] [--warmup 2] [--out profiles/r04_duplicate_match_b200.json]

Shapes: the configs[0] match (100 boards), the configs[3] match (65,536 boards) -- make_simple_duplicate_evaluate (host
loop: one host read of the live-row counts per step) against make_device_duplicate_evaluate (one brl_duplicate_match call).
Each timed call is a whole match, from the keys to the statistics on the host, between CUDA events; the two loops alternate
call by call after `warmup` calls of each, and every timed pair must give bit-equal per-env returns.  The card's name and
power limit are read in the same run.  The self-play league's former host loop was timed against its device loop here too:
profiles/r04_duplicate_match_b200.json (10 nets) and profiles/r09_league_host_vs_device_b200.json (10, 21 and 101 nets).
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.evaluation import make_device_duplicate_evaluate, make_simple_duplicate_evaluate  # noqa: E402
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


def compare(name, host_fn, dev_fn, returns_of, reps, warmup):
    for _ in range(warmup):
        host_fn()
        dev_fn()
    t_host, t_dev = [], []
    for _ in range(reps):
        th, rh = timed(host_fn)
        td, rd = timed(dev_fn)
        for a, b in zip(returns_of(rh), returns_of(rd)):
            if not torch.equal(a, b):
                raise SystemExit(f"{name}: device loop and host loop per-env returns differ")
        t_host.append(th)
        t_dev.append(td)
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    row = {"shape": name, "host_ms": t_host, "device_ms": t_dev, "host_median_ms": med(t_host), "device_median_ms": med(t_dev),
           "speedup": med(t_host) / med(t_dev), "bit_equal_cum_return": True}
    print(json.dumps({k: v for k, v in row.items() if not k.endswith("_ms") or "median" in k}))
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="profiles/r04_duplicate_match_b200.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    env = BridgeBidding(table=synthetic_deal_table(10_000, seed=1), device=dev)
    key = brandom.PRNGKey(0)
    rows = []
    nets = [seeded_params(900, dev), seeded_params(901, dev)]
    for n in (100, 65536):
        host = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)
        devm = make_device_duplicate_evaluate(env, "relu", "DeepMind", n)
        rows.append(compare(f"duplicate_match_{n}", lambda: host(nets[0], nets[1], key), lambda: devm(nets[0], nets[1], key),
                            lambda r: [r[3]], args.reps, args.warmup))
    result = {"card": card, "reps": args.reps, "warmup": args.warmup,
              "timing": "CUDA events around whole matches (keys to host statistics), loops alternating", "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"card": card, "out": args.out}))


if __name__ == "__main__":
    main()
