"""`train(config, rng)` of ppo.py:228-571 on the B200-native path: rollout -> GAE -> PPO
update per iteration, with the per-iteration strength probes, the FSP / PFSP opponent
league (ppo.py:392-470) and the DDS-table rotation (ppo.py:525-549).

Everything heavy runs in the kernels behind `brl_b200.ops`; this file is the control
plane only (config defaults, opponent selection, table rotation, logging hooks).  wandb,
OmegaConf and the dataset download are out of scope (SURVEY 2): `log_fn` receives the same
dict ppo.py would send to wandb, and `tables` are the deal tables to rotate through
(packed arrays or paths `deals.load_table` understands; synthetic when omitted, because the
DDS dataset cannot be downloaded offline).
"""
from __future__ import annotations

import os
import pickle
import time
from typing import Callable, Optional, Sequence

import numpy as np
import torch

from . import deals as _deals
from . import random as brandom
from .env import BridgeBidding
from .evaluation import (make_device_duplicate_evaluate, make_device_evaluate, make_device_pfsp_probe,
                         make_device_simple_evaluate, make_evaluate_log)
from .gae import make_calc_gae
from .models import LAYERS, ForwardPass, init_params, load_params, make_forward_pass
from .optim import make_optimizer
from .roll_out import make_roll_out
from .update import make_update_step
from .zoo import ModelZoo, device_zoo_fits


def default_config() -> dict:
    """PPOConfig defaults (ppo.py:117-182)."""
    return dict(
        seed=0, lr=0.000001, num_envs=8192, num_steps=32, total_timesteps=2_621_440_000, update_epochs=10,
        minibatch_size=1024, num_minibatches=128, num_updates=10000, dds_results_dir="dds_results", hash_size=100_000,
        num_eval_envs=10000, eval_opp_activation="relu", eval_opp_model_type="DeepMind", eval_opp_model_path=None,
        num_eval_step=10, save_model=True, save_model_interval=1, log_path="rl_log", exp_name="exp_0000",
        save_model_path="rl_params", track=False, load_initial_model=False, initial_model_path=None,
        actor_activation="relu", actor_model_type="DeepMind", game_mode="competitive", self_play=True,
        opp_activation="relu", opp_model_type="DeepMind", opp_model_path=None, ratio_model_zoo=0.0,
        num_model_zoo=100_000, threshold_model_zoo=-24.0, prioritized_fictitious=False, prior_t=0.1,
        num_prioritized_envs=100, gamma=1.0, gae_lambda=0.95, clip_eps=0.2, ent_coef=0.001, vf_coef=0.5,
        value_clipping=True, global_gradient_clipping=True, anneal_lr=False, reward_scaling=False, max_grad_norm=0.5,
        reward_scale=7600.0, actor_illegal_action_mask=True, actor_illegal_action_penalty=False,
        illegal_action_penalty=-1.0, illegal_action_l2norm_coef=0.0)


def params_to_host(params) -> dict:
    """haiku-layout dict of NumPy arrays (what ppo.py:351-362 pickles)."""
    return {name: {k: params[name][k].detach().cpu().numpy() for k in ("w", "b")} for name in LAYERS}


def save_params(params, path: str) -> None:
    with open(path, "wb") as fh:
        pickle.dump(params_to_host(params), fh)


def pfsp_probabilities(imp_list: np.ndarray, prior_t: float) -> np.ndarray:
    """ppo.py:437-449: softmax(-imp / T) over the zoo (harder opponents are sampled more)."""
    x = -np.asarray(imp_list, dtype=np.float64)
    e = np.exp((x - x.max()) / prior_t)
    return e / e.sum()


def make_evaluators(config: dict, eval_env, eval_opp_params):
    """The three evaluators of every iteration (ppo.py:252-283): (train/score vs eval_opp, the imp_opp / PFSP duplicate probe,
    the eval/* duplicate statistics), each a device loop of one brl_evaluate_match / brl_duplicate_match call.  They give
    the results of the host loops make_simple_evaluate / make_simple_duplicate_evaluate / make_evaluate."""
    act, mt = config["actor_activation"], config["actor_model_type"]
    opp_act, opp_mt = config["eval_opp_activation"], config["eval_opp_model_type"]
    return (make_device_simple_evaluate(eval_env, act, mt, opp_act, opp_mt, None, config["num_eval_envs"],
                                        team2_params=eval_opp_params),
            make_device_duplicate_evaluate(eval_env, act, mt, config["num_prioritized_envs"]),
            make_device_evaluate(eval_env, act, mt, opp_act, opp_mt, None, config["num_eval_envs"], config["game_mode"],
                                 duplicate=True, team2_params=eval_opp_params))


def train(config: dict, rng: int, tables: Optional[Sequence] = None, eval_table=None, device="cuda",
          log_fn: Optional[Callable[[dict], None]] = None, eval_opp_params=None, np_rng: Optional[np.random.Generator] = None,
          forward_pass_factory=None, update_step_factory=None):
    """`forward_pass_factory(activation, model_type)` / `update_step_factory(config, forward_pass, optimizer)` replace
    `make_forward_pass` / `make_update_step` -- the hook the cuBLAS cross-check (scripts/torch_baseline.py) plugs into;
    the defaults are the tensor-core kernels and nothing else."""
    make_fp = forward_pass_factory or make_forward_pass
    make_us = update_step_factory or make_update_step
    cfg = dict(default_config())
    cfg.update(config)
    config = cfg
    config["num_updates"] = config["total_timesteps"] // config["num_steps"] // config["num_envs"]   # ppo.py:225-227
    config["num_minibatches"] = config["num_envs"] * config["num_steps"] // config["minibatch_size"]  # ppo.py:228-230
    np_rng = np_rng or np.random.default_rng(config["seed"])
    dev = torch.device(device)

    def as_table(t):
        return _deals.load_table(t) if isinstance(t, str) else np.asarray(t, dtype=np.uint8)

    if tables is None:
        d = config["dds_results_dir"]
        if os.path.isdir(d):
            tables = [os.path.join(d, f) for f in sorted(os.listdir(d)) if "train" in f]            # ppo.py:292-294
            if eval_table is None and os.path.exists(os.path.join(d, "test_000.npy")):
                eval_table = os.path.join(d, "test_000.npy")                                      # ppo.py:252
        else:
            tables = [_deals.synthetic_deal_table(config["hash_size"], seed=config["seed"] + k) for k in range(2)]
    tables = [as_table(t) for t in tables]
    eval_table = as_table(eval_table) if eval_table is not None else _deals.synthetic_deal_table(config["hash_size"], seed=10_000)

    optimizer = make_optimizer(config)                                                            # ppo.py:195-211
    actor_forward_pass = make_fp(config["actor_activation"], config["actor_model_type"])
    rng, _rng = brandom.split(rng)
    params = init_params(_rng & 0x7FFFFFFF, dev)                                                  # ppo.py:240-243
    opt_state = optimizer.init(params)
    if config["load_initial_model"]:
        params = load_params(config["initial_model_path"], dev)                                   # ppo.py:246-248

    rng, eval_rng = brandom.split(rng)
    eval_env = BridgeBidding(table=eval_table, device=dev)
    if eval_opp_params is None:
        eval_opp_params = (load_params(config["eval_opp_model_path"], dev) if config["eval_opp_model_path"]
                           else init_params(12345, dev))
    simple_evaluate, simple_duplicate_evaluate, duplicate_evaluate = make_evaluators(config, eval_env, eval_opp_params)

    opp_forward_pass = make_fp(config["opp_activation"], config["opp_model_type"])
    envs = [BridgeBidding(table=t, device=dev) for t in tables]                                   # ppo.py:296-303
    roll_outs = [make_roll_out(config, env, actor_forward_pass, opp_forward_pass) for env in envs]
    calc_gae = make_calc_gae(config, actor_forward_pass)
    update_step = make_us(config, actor_forward_pass, optimizer)

    rng, _rng = brandom.split(rng)
    env, roll_out = envs[0], roll_outs[0]
    env_state = env.init(env.make_keys(_rng, config["num_envs"]))
    hash_index_list = np.arange(len(tables))
    steps, hash_index, board_count = 0, 0, 0
    terminated_count = torch.zeros((), dtype=torch.int64, device=dev)
    rng, _rng = brandom.split(rng)
    runner_state = (params, opt_state, env_state, env_state.observation, terminated_count, _rng)

    if not config["self_play"]:
        opp_params = load_params(config["opp_model_path"], dev) if config["opp_model_path"] else eval_opp_params
    else:
        opp_params = params
    # past models.  ppo.py keeps them on disk (params-XXXXXXXX.pkl under save_model_path) and loads one at a time; here they
    # only exist when the league can use them.  They are a zoo.ModelZoo packed in HBM (allocated once for every save the run
    # makes, up to num_model_zoo): the PFSP probe is one league call and an opponent one device copy.  If that pool does not
    # fit in free device memory at the start, or when the opponent's forward is not the tensor-core one (which reads a packed
    # opponent), they are host-memory NumPy dicts (14.7 MB each), copied to the device one at a time and probed one match
    # each.
    use_zoo = bool(config["self_play"]) and float(config["ratio_model_zoo"]) > 0.0
    zoo_capacity = min(config["num_model_zoo"], max(0, config["num_updates"] - 1) // config["save_model_interval"])
    zoo = []
    probe_envs = config["num_prioritized_envs"] if config["prioritized_fictitious"] else 0
    if use_zoo and isinstance(opp_forward_pass, ForwardPass) and device_zoo_fits(zoo_capacity, probe_envs, dev):
        zoo = ModelZoo(zoo_capacity, dev)
        if probe_envs:
            pfsp_probe = make_device_pfsp_probe(eval_env, config["actor_activation"], config["actor_model_type"], probe_envs)
            pfsp_probe.reserve(zoo)                          # all of the zoo's device memory is taken here, once
    device_zoo = isinstance(zoo, ModelZoo)

    def zoo_model(k: int):
        if device_zoo:
            return zoo.opponent(k)
        return {name: {kk: torch.as_tensor(v, device=dev) for kk, v in zoo[k][name].items()} for name in LAYERS}
    save_dir = os.path.join(config["log_path"], config["exp_name"], config["save_model_path"])
    if config["save_model"]:
        os.makedirs(save_dir, exist_ok=True)
    logs = []
    for i in range(config["num_updates"]):
        if i != 0 and i % config["save_model_interval"] == 0:                                      # ppo.py:351-362
            if device_zoo:
                zoo.append(runner_state[0])                  # keeps the newest zoo_capacity <= num_model_zoo models
            elif use_zoo:
                zoo.append(params_to_host(runner_state[0]))
                zoo[:] = zoo[-config["num_model_zoo"]:]
            if config["save_model"]:
                save_params(runner_state[0], os.path.join(save_dir, f"params-{i:08}.pkl"))
        t0 = time.time()
        R = simple_evaluate(runner_state[0], eval_rng)                                            # ppo.py:365-368
        eval_log = {}
        if i % config["num_eval_step"] == 0:                                                      # ppo.py:369-374
            log_info, _, _ = duplicate_evaluate(runner_state[0], eval_rng)
            eval_log = make_evaluate_log(log_info)
        t_eval = time.time() - t0

        if config["self_play"]:                                                                   # ppo.py:376-470
            (imp_opp, _, _), _, _, _ = simple_duplicate_evaluate(runner_state[0], opp_params, eval_rng)
            if imp_opp >= config["threshold_model_zoo"]:
                if len(zoo) != 0 and np_rng.binomial(1, config["ratio_model_zoo"]):
                    if config["prioritized_fictitious"]:
                        imp_list = np.zeros(len(zoo))
                        if device_zoo:  # the learner against every zoo model in one league call
                            imp_list[:] = [imp for imp, _, _ in pfsp_probe(runner_state[0], zoo, eval_rng)]
                        else:
                            for k in range(len(zoo)):  # one past model on the device at a time
                                (imp_list[k], _, _), _, _, _ = simple_duplicate_evaluate(runner_state[0], zoo_model(k),
                                                                                         eval_rng)
                        opp_params = zoo_model(int(np_rng.choice(len(zoo), p=pfsp_probabilities(imp_list, config["prior_t"]))))
                    else:
                        opp_params = zoo_model(int(np_rng.integers(len(zoo))))
                else:
                    opp_params = runner_state[0]
        (imp_opp_before, _, _), _, _, _ = simple_duplicate_evaluate(runner_state[0], opp_params, eval_rng)
        torch.cuda.synchronize(dev)
        t1 = time.time()
        runner_state, traj_batch = roll_out(runner_state, opp_params)                             # ppo.py:472-475
        torch.cuda.synchronize(dev)
        t2 = time.time()
        advantages, targets = calc_gae(runner_state, traj_batch)                                  # ppo.py:477
        torch.cuda.synchronize(dev)
        t3 = time.time()
        runner_state, loss_info = update_step(runner_state, traj_batch, advantages, targets)     # ppo.py:479-484
        torch.cuda.synchronize(dev)
        t4 = time.time()
        (imp_opp_after, _, _), _, _, _ = simple_duplicate_evaluate(runner_state[0], opp_params, eval_rng)
        steps += config["num_envs"] * config["num_steps"]
        total_loss, (value_loss, loss_actor, entropy, approx_kl, clipflacs, illegal_action_loss) = loss_info
        lr_now = optimizer.lr_at((i + 1) * config["update_epochs"] * config["num_minibatches"])
        board_num = int(runner_state[4])
        log = {                                                                                   # ppo.py:508-523
            "train/score": float(R), "train/total_loss": float(total_loss[-1][-1]),
            "train/value_loss": float(value_loss[-1][-1]), "train/loss_actor": float(loss_actor[-1][-1]),
            "train/illegal_action_loss": float(illegal_action_loss[-1][-1]), "train/policy_entropy": float(entropy[-1][-1]),
            "train/clipflacs": float(clipflacs[-1][-1]), "train/approx_kl": float(approx_kl[-1][-1]), "train/lr": lr_now,
            "train/imp_opp_before": float(imp_opp_before), "train/imp_opp_after": float(imp_opp_after),
            "board_num": board_num, "steps": steps,
            "time/eval": t_eval, "time/rollout": t2 - t1, "time/calc_gae": t3 - t2, "time/update": t4 - t3,
        }
        log.update(eval_log)
        logs.append(log)
        if log_fn is not None:
            log_fn(log)
        if (board_num - board_count) // config["hash_size"] >= 1:                                 # ppo.py:525-549
            hash_index += 1
            board_count = board_num
            if hash_index == len(hash_index_list):
                hash_index = 0
                np_rng.shuffle(hash_index_list)
            env, roll_out = envs[hash_index_list[hash_index]], roll_outs[hash_index_list[hash_index]]
            rng, _rng = brandom.split(rng)
            env_state = env.init(env.make_keys(_rng, config["num_envs"]))
            runner_state = (runner_state[0], runner_state[1], env_state, env_state.observation, runner_state[4], _rng)
            log["table"] = int(hash_index_list[hash_index])
    if config["save_model"]:                                                                      # ppo.py:550-569
        save_params(runner_state[0], os.path.join(save_dir, f"params-{config['num_updates']:08}.pkl"))
        with open(os.path.join(save_dir, f"opt_state-{config['num_updates']:08}.pkl"), "wb") as fh:
            st = runner_state[1]
            pickle.dump({"count": st.count, "mu": st.mu.cpu().numpy(), "nu": st.nu.cpu().numpy()}, fh)
    return runner_state, logs
