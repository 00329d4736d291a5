"""Cost of the bidding-system statistics on the GPU (DESIGN.md f15).

    python scripts/bidding_system_bench.py [--out profiles/r17_system_b200.json] [--reps 7]

- A self-play match (one net on all four seats, brl_duplicate_match) at 100, 10,000 and 65,536 boards, with and without
  the histogram [21], the two alternating rep by rep; CUDA events around each call, after one warm-up call of each (which
  captures its graph).
- brl_system_stats_auctions on the 2,000 golden auctions tiled to about 1M, as auctions/s.
Medians and ranges over the reps; the card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, ops, random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.evaluation import _MatchBuffers  # noqa: E402
from brl_b200.models import init_params, make_forward_pass  # noqa: E402

DEV = "cuda:0"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def _timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def _stats(xs):
    return dict(median_ms=float(np.median(xs)), min_ms=float(np.min(xs)), max_ms=float(np.max(xs)))


def match_leg(env, n, reps):
    fp = make_forward_pass("relu", "DeepMind")
    b = _MatchBuffers(n, 1, 0, DEV, with_models=True, with_tables=False)
    fp.pack_into(init_params(3, DEV), b.pool[0, :ops._lib.load().brl_mlp_packed_bytes()])
    _, sub = brandom.split(brandom.PRNGKey(0))
    b.keys.copy_(env.make_keys(sub, n))
    b.env_models.zero_()
    hist = ops.new_system_hist(1, DEV)
    play = {"plain": lambda: b.play(env, False, 0), "hist": lambda: b.play(env, False, 0, hist)}
    for f in play.values():
        f()
    torch.cuda.synchronize()
    times = {k: [] for k in play}
    for _ in range(reps):
        for k, f in play.items():
            times[k].append(_timed(f))
    decisions = int(ops.system_hist_counts(hist)[..., 95].sum()) // (reps + 1)
    out = {k: _stats(v) for k, v in times.items()}
    out["overhead_of_median"] = out["hist"]["median_ms"] / out["plain"]["median_ms"] - 1.0
    out["decisions_per_match"] = decisions
    return out


def auctions_leg(reps):
    z = np.load(os.path.join(GOLDEN, "auctions.npz"))
    table = torch.as_tensor(np.load(os.path.join(GOLDEN, "boards_wb5_1000.npz"))["table"], device=DEV)
    tiles = 500
    lens = np.diff(z["offsets"]).astype(np.int64)
    lens = np.tile(lens, tiles)
    offsets = torch.as_tensor(np.concatenate([[0], np.cumsum(lens)]), device=DEV)
    calls = torch.as_tensor(np.tile(z["calls"].astype(np.uint8), tiles), device=DEV)
    board = torch.as_tensor(np.tile(z["board"].astype(np.int32), tiles), device=DEV)
    dealer = torch.as_tensor(np.tile(z["dealer"].astype(np.int8), tiles), device=DEV)
    hist = ops.new_system_hist(1, DEV)
    n = len(lens)

    def run():
        hist.view(torch.int32).zero_()
        ops._call("brl_system_stats_auctions", [ops._ptr(table), ops._ptr(calls), ops._ptr(offsets), ops._ptr(board),
                                                ops._ptr(dealer), ops._ptr(hist)], ops._params(n, n_deals=table.shape[0]))

    ops.system_stats_auctions(table, calls, offsets, hist, board=board, dealer=dealer)   # the checked call, once
    run()
    torch.cuda.synchronize()
    t = [_timed(run) for _ in range(reps)]
    med = float(np.median(t))
    return dict(auctions=n, calls=int(lens.sum()), **_stats(t), auctions_per_s=n / (med * 1e-3),
                note="kernel plus a 1.09 MB histogram memset per timed call; the host checks of the op wrapper run once, untimed")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r17_system_b200.json")
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    card = _card()
    env = BridgeBidding(table=synthetic_deal_table(100_000, seed=0), device=DEV)
    res = dict(card=card, reps=args.reps, method="CUDA events around each call; plain and histogram calls alternate",
               match={str(n): match_leg(env, n, args.reps) for n in (100, 10_000, 65_536)}, auctions=auctions_leg(args.reps),
               card_after=_card())
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
