"""Self-play league timing (workspace/eval_selfplay_league.py): the batched tournament over M seeded nets against the
pairwise make_simple_duplicate_evaluate loop.

    python scripts/selfplay_league_bench.py [--models 21 101] [--pairwise-models 21] [--boards 100] [--out FILE]

Per M: wall time of league(params_list, rng) (CUDA-synchronised host clock, after one warm-up league on the same M) and
the pool's bytes.  For --pairwise-models the pairwise loop is timed too and its matrices must equal the league's.  The
card's name and power limit are read in the same process.  Writes one JSON object (stdout and --out).
"""
import argparse
import itertools
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, evaluation, ops, random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.models import init_params, LAYERS  # noqa: E402


def seeded(seed, dev):  # tests/helpers.seeded_params: trained-size logits, so decisions are not near-ties
    p = init_params(seed, dev)
    p[LAYERS[4]]["w"] *= 128
    return p


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return [s.strip() for s in q.split(",")]
    except Exception as exc:  # noqa: BLE001
        return [torch.cuda.get_device_name(0), f"power limit unknown ({exc})"]


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--models", type=int, nargs="+", default=[21, 101])
    ap.add_argument("--pairwise-models", type=int, nargs="*", default=[21])
    ap.add_argument("--boards", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    name, *power = card()
    env = BridgeBidding(table=synthetic_deal_table(10_000, seed=0), device=dev)
    key = brandom.PRNGKey(0)
    league = evaluation.make_selfplay_league_evaluate(env, "relu", "DeepMind", a.boards)
    res = {"gpu": name, "power_limit_and_max_sm_clock": power, "boards_per_match": a.boards, "runs": []}
    for M in a.models:
        nets = [seeded(1000 + m, dev) for m in range(M)]
        league(nets, key)                                                  # warm-up: kernels, tensor maps, allocator
        t_league, (stats, wl, dis, clip) = timed(lambda: league(nets, key))
        run = {"models": M, "matches": len(stats), "boards": len(stats) * a.boards, "league_s": t_league,
               "pool_bytes": M * ops.mlp_pool_stride()}
        if M in a.pairwise_models:
            match = evaluation.make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", a.boards)
            pairs = list(itertools.combinations(range(M), 2))
            match(nets[0], nets[1], key)                                   # warm-up

            def pairwise():
                return {p: match(nets[p[0]], nets[p[1]], key)[0] for p in pairs}
            t_pair, pstats = timed(pairwise)
            mats = evaluation.league_matrices(M, {p: s[0] for p, s in pstats.items()})
            run["pairwise_s"] = t_pair
            run["speedup"] = t_pair / t_league
            run["matrices_identical"] = all(np.array_equal(x, y) for x, y in zip(mats, (wl, dis, clip)))
            run["max_stat_rel_diff"] = max(abs(s - q) / max(abs(q), 1e-300) for p in pairs
                                           for s, q in zip(stats[p], pstats[p]))
        res["runs"].append(run)
        print(json.dumps(run), flush=True)
        del nets
        torch.cuda.empty_cache()
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
