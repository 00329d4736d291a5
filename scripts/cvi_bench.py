"""Cost of call-value policy improvement on the GPU (DESIGN.md f17).

    python scripts/cvi_bench.py [--out profiles/r19_cvi_b200.json] [--reps 5]

  call_values   one brl_call_values call (self-play, an `init_params` net on all four seats) at 1,000 and 10,000 boards with
                the eight records, without and with the training examples [19] / [20], alternating rep by rep
  step          one brl_cv_grad + brl_mlp_adam_step at B = 1,024 and 8,192 (bf16 observations, clipping on)
  iteration     one cvi.train iteration at boards_per_iter = 10,000 (collect + update, no evaluation, lr = 0), over
                iterations 2 .. reps + 1 of one run
CUDA events around each call after a warm-up call of each shape (which captures the match graphs).  Medians and ranges
over the reps; the card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, cvi, ops, random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.evaluation import _MatchBuffers  # noqa: E402
from brl_b200.models import init_params, make_forward_pass  # noqa: E402
from scripts.call_values_bench import _card, _stats, _timed  # noqa: E402

DEV = "cuda:0"


def call_values_leg(env, n, reps):
    fp = make_forward_pass("relu", "DeepMind")
    b = _MatchBuffers(n, 1, 0, DEV, with_models=True, with_tables=True)
    fp.pack_into(init_params(3, DEV), b.pool[0, :ops._lib.load().brl_mlp_packed_bytes()])
    _, sub = brandom.split(brandom.PRNGKey(0))
    b.keys.copy_(env.make_keys(sub, n))
    b.env_models.zero_()
    b.play(env, False, 0)
    scratch = torch.empty(ops.call_values_scratch_bytes(n, 1), dtype=torch.uint8, device=DEV)
    gain = torch.empty((1,) + ops.CALL_GAIN_SHAPE, dtype=torch.int64, device=DEV)
    regret = torch.empty((1,) + ops.CALL_REGRET_SHAPE, dtype=torch.int64, device=DEV)
    mismatch = torch.empty(1, dtype=torch.int64, device=DEV)
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    recs = {"records": ops.CallValueRecords(48 * n, DEV), "records_and_examples": ops.CallValueRecords(48 * n, DEV, True)}
    play = {k: (lambda r=r: ops.call_values(b.keys, env.table, b.pool, b.env_models, b.tables[0].rewards, b.tables[1].rewards,
                                            scratch, gain, regret, mismatch, status, records=r)) for k, r in recs.items()}
    for f in play.values():
        f()
    torch.cuda.synchronize()
    assert int(status[0]) == 0
    times = {k: [] for k in play}
    for _ in range(reps):
        for k, f in play.items():
            times[k].append(_timed(f))
    out = {k: _stats(v) for k, v in times.items()}
    out["ratio_of_medians"] = out["records_and_examples"]["median_ms"] / out["records"]["median_ms"]
    out["decisions"] = int(recs["records"].count[0])
    return out


def step_leg(B, reps):
    params = init_params(5, DEV)
    upd = cvi.Updater(dict(cvi.default_config(), minibatch_size=B), params, DEV)
    g = torch.Generator(device="cpu").manual_seed(B)
    obs = (torch.rand((B, ops.OBS_DIM), generator=g) < 0.05).to(torch.bfloat16).to(DEV)
    gain = torch.randint(-12, 13, (B, ops.NUM_ACTIONS), generator=g).float()
    gain[torch.rand((B, ops.NUM_ACTIONS), generator=g) < 0.6] = float("nan")
    gain[:, 0] = 0.0
    gain = gain.to(DEV)
    stats = torch.zeros(8, device=DEV)

    def step():
        ops.cv_grad(obs, upd.blob, upd.scratch, gain, upd.grads, stats, upd.acc, ent_coef=0.001)
        upd.opt_state = upd.optimizer.update_mlp_(upd.flat, upd.grads, upd.opt_state, upd.acc[14:15], upd.blob)
    step()
    torch.cuda.synchronize()
    return _stats([_timed(step) for _ in range(max(reps, 20))])


def iteration_leg(table, reps):
    """iterations 2 .. reps + 1 of one cvi.train run (the first captures the match graphs): time/collect and time/update,
    host clocks around work that ends in a device synchronise.  lr = 0 (the Adam step still runs): the cost follows the
    number of decisions, and trained from a random net the play changes within a few iterations (toward passed-out
    boards), so every timed iteration plays the same net instead."""
    cfg = dict(boards_per_iter=10_000, num_iters=reps + 1, epochs=1, minibatch_size=1024, num_eval_envs=100,
               num_eval_step=1 << 30, save_model=False, lr=0.0)
    _, logs = cvi.train(cfg, 0, table, device=DEV)
    logs = logs[1:]
    out = {k: _stats([1e3 * lg[f"time/{k}"] for lg in logs]) for k in ("collect", "update")}
    out["iteration"] = _stats([1e3 * (lg["time/collect"] + lg["time/update"]) for lg in logs])
    out["decisions"] = [lg["cv/decisions"] for lg in logs]
    out["minibatches"] = [lg["cv/decisions"] // 1024 for lg in logs]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r19_cvi_b200.json")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    table = synthetic_deal_table(100_000, seed=1)
    env = BridgeBidding(table=table, device=DEV)
    res = {"card": _card(), "reps": a.reps,
           "call_values": {str(n): call_values_leg(env, n, a.reps) for n in (1000, 10_000)},
           "step": {str(B): step_leg(B, a.reps) for B in (1024, 8192)},
           "iteration_10000_boards": iteration_leg(table, a.reps)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
