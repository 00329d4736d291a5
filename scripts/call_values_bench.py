"""Cost of the counterfactual call values on the GPU (DESIGN.md f16).

    python scripts/call_values_bench.py [--out profiles/r18_call_values_b200.json] [--reps 5]

One brl_call_values call (self-play: one net on all four seats, `init_params` nets) at 100, 1,000 and 10,000 boards with
M = 1 and M = 4 (board blocks of the four nets, as make_call_values_evaluate lays them out), against the base match alone
(brl_duplicate_match on the same envs), the two alternating rep by rep; CUDA events around each call after one warm-up call
of each (which captures its graph).  Beside each time: decisions and branch rows (legal alternatives) per board, and the
unpinned forward's `mismatch` count.  At 100 boards the host-loop reference (tests/call_values_ref.py) is timed once.
Medians and ranges over the reps; the card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, ops, random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.evaluation import _MatchBuffers  # noqa: E402
from brl_b200.models import init_params, make_forward_pass  # noqa: E402

DEV = "cuda:0"


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


def leg(env, boards, M, reps):
    n = boards * M
    fp = make_forward_pass("relu", "DeepMind")
    b = _MatchBuffers(n, M, 0, DEV, with_models=True, with_tables=True)
    size = ops._lib.load().brl_mlp_packed_bytes()
    for m in range(M):
        fp.pack_into(init_params(3 + m, DEV), b.pool[m, :size])
    _, sub = brandom.split(brandom.PRNGKey(0))
    b.keys.copy_(env.make_keys(sub, boards).repeat(M))
    b.env_models.copy_(torch.arange(M, dtype=torch.int32, device=DEV).repeat_interleave(boards)[:, None].expand(n, 2))
    scratch = torch.empty(ops.call_values_scratch_bytes(n, M), dtype=torch.uint8, device=DEV)
    gain = torch.empty((M,) + ops.CALL_GAIN_SHAPE, dtype=torch.int64, device=DEV)
    regret = torch.empty((M,) + ops.CALL_REGRET_SHAPE, dtype=torch.int64, device=DEV)
    mismatch = torch.empty(M, dtype=torch.int64, device=DEV)
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    ra, rb = b.tables[0].rewards, b.tables[1].rewards
    play = {"base_match": lambda: b.play(env, False, 0),
            "call_values": lambda: ops.call_values(b.keys, env.table, b.pool, b.env_models, ra, rb, scratch, gain, regret,
                                                   mismatch, status, illegal_penalty=env.illegal_penalty,
                                                   illegal_bonus=env.illegal_bonus)}
    for f in play.values():
        f()
    torch.cuda.synchronize()
    assert int(status[0]) == 0 and int(b.status[0]) == 0
    times = {k: [] for k in play}
    for _ in range(reps):
        for k, f in play.items():
            times[k].append(_timed(f))
    out = {k: _stats(v) for k, v in times.items()}
    out["ratio_of_medians"] = out["call_values"]["median_ms"] / out["base_match"]["median_ms"]
    out["decisions_per_board"] = int(regret[..., 0].sum()) / n
    out["branch_rows_per_board"] = int(gain[..., 0].sum()) / n
    out["mismatch_unpinned"] = int(mismatch.sum())
    out["forward_rows_per_board"] = "not counted"
    return out


def host_leg(env):
    from tests import call_values_ref as R
    nets = [init_params(3, DEV)]
    t0 = time.perf_counter()
    rec, _, _ = R.host_records(env, nets, (0, 0), 100, brandom.PRNGKey(100))
    torch.cuda.synchronize()
    return dict(boards=100, seconds=time.perf_counter() - t0, decisions=len(rec["env"]),
                note="tests/call_values_ref.py host loop, one run, M = 1")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r18_call_values_b200.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default="100,1000,10000")
    args = ap.parse_args()
    card = _card()
    env = BridgeBidding(table=synthetic_deal_table(100_000, seed=0), device=DEV)
    res = dict(card=card, reps=args.reps, method="CUDA events around each call; base match and call values alternate",
               legs={f"{s}x{M}": leg(env, s // M if M > 1 else s, M, args.reps) for s in map(int, args.sizes.split(","))
                     for M in (1, 4)},
               host_reference=host_leg(env), card_after=_card())
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
