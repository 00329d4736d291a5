"""Call-value iteration (DESIGN.md f17): train a net on the IMPs each legal call would have won.

Each iteration plays `boards_per_iter` fresh boards with brl_call_values (DESIGN.md f16): at every decision of the learner,
every legal call is played out by the nets themselves, so the decision's gains g(a) are the value of calling a there
against the current play, in IMPs.  The update maximises sum_a pi(a | obs) g(a) -- an all-actions policy-gradient step with
one exact value per legal call -- through `brl_cv_grad` (the tensor-core forward / backward with the loss head of
include/brl_b200.h) and `brl_mlp_adam_step`.  It does not train toward argmax_a g(a), the hindsight regret of f16.

    params, logs = cvi.train(cfg, rng=0, table=deal_table)

Self-play (`opponent_model_path` None) puts the learner in all four seats.  With an opponent, the learner plays players
0/1 against the fixed net on 2/3, and only the learner's decisions are trained on.  Parameters are saved with
ppo.save_params, so ppo.train loads them as `initial_model_path` and cvi.train loads ppo's.  One GPU only: the evaluator
shards boards across ranks, and a driver on several ranks would train each on its own shard.
"""
from __future__ import annotations

import math
import os
import time
from typing import Callable, Optional

import numpy as np
import torch

from . import deals as _deals
from . import dist as bdist
from . import ops
from . import random as brandom
from .env import BridgeBidding
from .evaluation import make_call_values_evaluate, make_device_duplicate_evaluate
from .models import check_params_file, init_params, load_params
from .optim import flatten_params, make_optimizer
from .ppo import save_params

STAT_KEYS = ("cv/total_loss", "cv/mean_gain", "cv/argmax_gain", "cv/argmax_regret", "cv/entropy", "cv/argmax_best",
             "cv/illegal_prob")  # brl_cv_grad's stats 0..6
SIZE_KEYS = ("boards_per_iter", "num_iters", "epochs", "minibatch_size", "num_eval_envs", "num_eval_step",
             "save_model_interval")


def default_config() -> dict:
    return dict(lr=1e-6, ent_coef=0.001, max_grad_norm=0.5, boards_per_iter=10_000, num_iters=100, epochs=1,
                minibatch_size=1024, seed=0, initial_model_path=None, opponent_model_path=None, eval_opp_model_path=None,
                num_eval_envs=10_000, num_eval_step=10, save_model=True, save_model_interval=10, log_path="cvi_log",
                exp_name="exp_0000")


def check_config(cfg: dict) -> None:
    """ValueError for a non-positive size, a negative or non-finite lr / ent_coef / max_grad_norm, a model file that is not a
    DeepMind 4x1024 set (read on the host only) and a process group of more than one rank"""
    for k in SIZE_KEYS:
        v = cfg[k]
        if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or v <= 0:
            raise ValueError(f"cvi: {k} must be a positive integer; got {v!r}")
    for k in ("lr", "ent_coef", "max_grad_norm"):
        v = cfg[k]
        if isinstance(v, bool) or not isinstance(v, (int, float, np.integer, np.floating)) or not math.isfinite(v) or v < 0:
            raise ValueError(f"cvi: {k} must be a finite number >= 0; got {v!r}")
    for k in ("initial_model_path", "opponent_model_path", "eval_opp_model_path"):
        if cfg[k]:
            check_params_file(cfg[k])
    _, world = bdist.rank_world()
    if world > 1:
        raise ValueError(f"cvi.train runs on one GPU: the process group has {world} ranks (the evaluator would shard the "
                         "boards and each rank would train on its own shard)")


def iteration_key(seed: int, iteration: int) -> int:
    """the board key of iteration `iteration`: fresh boards every iteration, the same for the same (seed, iteration)"""
    return brandom.PRNGKey(brandom.PRNGKey(seed) + iteration)


def permutation_generator(seed: int, iteration: int) -> torch.Generator:
    """the host generator of iteration `iteration`'s minibatch permutations (one randperm per epoch)"""
    return torch.Generator().manual_seed(int(iteration_key(seed ^ 0x5045524D, iteration) & 0x7FFFFFFFFFFFFFFF))


class Updater:
    """The update loop on fixed-address buffers: `epochs` passes of shuffled minibatches of brl_cv_grad + brl_mlp_adam_step
    over one set of device examples (the ragged last minibatch dropped, as ppo does).  The per-minibatch stats stay on the
    device until `run` returns them."""

    def __init__(self, cfg: dict, params, dev):
        self.cfg, self.dev = cfg, dev
        self.flat, self.views = flatten_params(params)
        self.blob = ops.mlp_pack_train(self.flat)
        self.optimizer = make_optimizer(dict(lr=float(cfg["lr"]), max_grad_norm=float(cfg["max_grad_norm"])))
        self.opt_state = self.optimizer.init(self.views)
        self.grads = torch.empty_like(self.flat)
        mb = int(cfg["minibatch_size"])
        self.scratch = ops.mlp_train_scratch(mb, dev)
        self.acc = ops.sl_acc(dev)
        self.obs = torch.empty((mb, ops.OBS_DIM), dtype=torch.bfloat16, device=dev)
        self.gain = torch.empty((mb, ops.NUM_ACTIONS), dtype=torch.float32, device=dev)

    def run(self, obs: torch.Tensor, gain: torch.Tensor, generator: torch.Generator) -> torch.Tensor:
        """-> device stats float32[epochs, minibatches, 8]"""
        cfg = self.cfg
        mb, epochs = int(cfg["minibatch_size"]), int(cfg["epochs"])
        n = int(gain.shape[0])
        nmb = n // mb
        stats = torch.zeros((epochs, nmb, 8), dtype=torch.float32, device=self.dev)
        ent = float(cfg["ent_coef"])
        for e in range(epochs):
            perm = torch.randperm(n, generator=generator).to(torch.int32).to(self.dev)
            for k in range(nmb):
                idx = perm[k * mb:(k + 1) * mb]
                ops.gather_rows(obs, idx, self.obs)
                ops.gather_rows(gain, idx, self.gain)
                ops.cv_grad(self.obs, self.blob, self.scratch, self.gain, self.grads, stats[e, k], self.acc, ent_coef=ent)
                self.opt_state = self.optimizer.update_mlp_(self.flat, self.grads, self.opt_state, self.acc[14:15], self.blob)
        return stats


def train(config: dict, rng: int, table, eval_table=None, device="cuda", log_fn: Optional[Callable[[dict], None]] = None,
          eval_opp_params=None):
    """Call-value iteration for `num_iters` iterations on boards of `table` (a packed deal table or a path
    deals.load_table reads).  `seed` keys the initial net when there is no initial_model_path (models.init_params), the
    boards and the minibatch order; `rng` seeds the eval opponent when neither eval_opp_params nor eval_opp_model_path
    gives one.  `log_fn(log)` receives per iteration:
    cv/decisions (examples trained on), cv/mean_regret (f16's mean regret of the learner's decisions), the last epoch's
    means of brl_cv_grad's stats 0..6 (STAT_KEYS) and every epoch's under the same key + "_epochs", time/collect,
    time/update, and every num_eval_step iterations eval/imp and eval/imp_se (the learner against the eval opponent,
    make_device_duplicate_evaluate on num_eval_envs boards of eval_table).  Saves log_path/exp_name/params-{iteration:08}.pkl
    every save_model_interval iterations and at the end.  -> (params, logs)."""
    cfg = default_config()
    unknown = set(config) - set(cfg)
    if unknown:
        raise ValueError(f"cvi: unknown config keys {sorted(unknown)}")
    cfg.update(config)
    check_config(cfg)
    dev = torch.device(device)
    as_table = lambda t: _deals.load_table(t) if isinstance(t, str) else np.asarray(t, dtype=np.uint8)  # noqa: E731
    env = BridgeBidding(table=as_table(table), device=dev)
    eval_env = BridgeBidding(table=as_table(eval_table) if eval_table is not None
                             else _deals.synthetic_deal_table(max(cfg["num_eval_envs"], 1000), seed=10_000), device=dev)
    params = load_params(cfg["initial_model_path"], dev) if cfg["initial_model_path"] else init_params(int(cfg["seed"]), dev)
    upd = Updater(cfg, params, dev)
    opponent = load_params(cfg["opponent_model_path"], dev) if cfg["opponent_model_path"] else None
    if eval_opp_params is None:
        eval_opp_params = (load_params(cfg["eval_opp_model_path"], dev) if cfg["eval_opp_model_path"]
                           else init_params(int(rng) & 0x7FFFFFFF, dev))
    collect = make_call_values_evaluate(env, "relu", "DeepMind", int(cfg["boards_per_iter"]))
    evaluate = make_device_duplicate_evaluate(eval_env, "relu", "DeepMind", int(cfg["num_eval_envs"]))
    save_dir = os.path.join(cfg["log_path"], cfg["exp_name"])
    if cfg["save_model"]:
        os.makedirs(save_dir, exist_ok=True)
    seed, logs = int(cfg["seed"]), []
    eval_key = brandom.PRNGKey(seed ^ 0x4556414C)              # the same eval boards at every evaluation
    for i in range(int(cfg["num_iters"])):
        torch.cuda.synchronize(dev)
        t0 = time.time()
        key = iteration_key(seed, i)
        if opponent is None:                                  # self-play: the learner in all four seats
            out = collect([upd.views], key, records="train")
            obs, gain = out["examples"]["obs"], out["examples"]["gain"]
        else:                                                 # the learner on players 0/1, the opponent on 2/3
            out = collect([upd.views, opponent], key, records="train", matches=[(0, 1)])
            mine = out["examples"]["net"] == 0
            obs, gain = out["examples"]["obs"][mine].contiguous(), out["examples"]["gain"][mine].contiguous()
        torch.cuda.synchronize(dev)
        t1 = time.time()
        stats = upd.run(obs, gain, permutation_generator(seed, i))
        torch.cuda.synchronize(dev)
        t2 = time.time()
        regret = out["regret_sums"][0]
        decisions = int(regret[:, 0].sum())
        log = {"cv/decisions": int(gain.shape[0]),
               "cv/mean_regret": float(regret[:, 1].sum()) / decisions if decisions else float("nan")}
        host = stats.cpu().numpy().astype(np.float64)
        by_epoch = host.mean(axis=1) if host.shape[1] else np.full((host.shape[0], 8), np.nan)
        for k, name in enumerate(STAT_KEYS):
            log[name] = float(by_epoch[-1, k])
            log[name + "_epochs"] = [float(x) for x in by_epoch[:, k]]
        log["time/collect"], log["time/update"] = t1 - t0, t2 - t1
        if i % int(cfg["num_eval_step"]) == 0:
            (imp, se, _), _, _, _ = evaluate(upd.views, eval_opp_params, eval_key)
            log["eval/imp"], log["eval/imp_se"] = float(imp), float(se)
        logs.append(log)
        if log_fn is not None:
            log_fn(log)
        if cfg["save_model"] and (i + 1) % int(cfg["save_model_interval"]) == 0:
            save_params(upd.views, os.path.join(save_dir, f"params-{i + 1:08}.pkl"))
    if cfg["save_model"]:
        save_params(upd.views, os.path.join(save_dir, f"params-{int(cfg['num_iters']):08}.pkl"))
    return upd.views, logs
