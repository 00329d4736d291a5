"""`train(config, rng)` of ppo.py:228-571 on the B200-native path: rollout -> GAE -> PPO
update per iteration, with the per-iteration strength probes, the FSP / PFSP opponent
league (ppo.py:392-470) and the DDS-table rotation (ppo.py:525-549).

KL anchor (not in the reference): `anchor_model_path` names a fixed net of the actor's architecture (e.g. the SL model a
run starts from) and `anchor_kl_coef` the weight of coef * mean KL(policy || anchor) in every minibatch's loss.  The
roll-out records the anchor's logits, the update adds the term (a loss term: rewards, GAE and value targets are
unchanged), and the log gains `train/anchor_kl`.  Unset (the default), every code path is the one without the feature.

Double-dummy par (not in the reference; DESIGN.md f13): `reward_mode="par_imp"` trains on IMP(score - par) / 24 instead of
score / reward_scale (roll_out.py), and `log_par=True` adds eval/imp_vs_par, eval/abs_imp_vs_par and eval/par_contract_rate
of the eval/* duplicate match to the iterations that play it (evaluation.par_statistics).  The defaults ("score", False)
leave every code path as it was.

Fixed partner (not in the reference; DESIGN.md f14): `partner_model_path` names a DeepMind 4x1024 net that bids as the
learner's partner.  It plays the roll-out's sub-step 3 (the partner slot of the quad step) and is team 1's partner in
train/score, the imp_opp_before / imp_opp_after probes and the eval/* match (log_par's too); the opponent team stays
(opp, opp) and the partner is not trained.  Unset (the default), every code path is the one without the feature.

Everything heavy runs in the kernels behind `brl_b200.ops`; this file is the control
plane only (config defaults, opponent selection, table rotation, logging hooks).  wandb,
OmegaConf and the dataset download are out of scope (SURVEY 2): `log_fn` receives the same
dict ppo.py would send to wandb, and `tables` are the deal tables to rotate through
(packed arrays or paths `deals.load_table` understands; synthetic when omitted, because the
DDS dataset cannot be downloaded offline).
"""
from __future__ import annotations

import math
import os
import pickle
import time
from typing import Callable, Optional, Sequence

import numpy as np
import torch

from . import deals as _deals
from . import pbt as _pbt
from . import random as brandom
from .env import BridgeBidding
from .evaluation import (make_device_duplicate_evaluate, make_device_evaluate, make_device_pfsp_probe,
                         make_device_simple_evaluate, make_evaluate_log, par_statistics)
from .gae import make_calc_gae
from .models import LAYERS, ForwardPass, check_params_file, init_params, load_params, make_forward_pass
from .optim import OptState, make_optimizer
from .pbt import default_pbt_config  # noqa: F401 -- ppo.default_pbt_config(): the options of train_population's `pbt`
from .roll_out import check_reward_mode, make_roll_out
from .update import check_population_configs, make_population_update_step, make_update_step
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
        illegal_action_penalty=-1.0, illegal_action_l2norm_coef=0.0, anchor_model_path=None, anchor_kl_coef=0.0,
        reward_mode="score", log_par=False, partner_model_path=None)


def check_anchor_config(config: dict) -> None:
    """ValueError for an anchor_kl_coef that is negative or not a finite number, or non-zero without anchor_model_path"""
    coef = config.get("anchor_kl_coef", 0.0)
    if isinstance(coef, bool) or not isinstance(coef, (int, float, np.integer, np.floating)) or not math.isfinite(coef) or coef < 0:
        raise ValueError(f"anchor_kl_coef must be a finite number >= 0; got {coef!r}")
    if coef != 0 and not config.get("anchor_model_path"):
        raise ValueError(f"anchor_kl_coef = {coef!r} needs an anchor net: set anchor_model_path")


def check_partner_config(config: dict) -> None:
    """ValueError for a partner_model_path together with ratio_model_zoo > 0 (zoo opponents have no partner slot), and for a
    file that is not a DeepMind 4x1024 parameter set; reads the file on the host only"""
    path = config.get("partner_model_path")
    if not path:
        return
    if float(config.get("ratio_model_zoo", 0.0)) > 0.0:
        raise ValueError("partner_model_path cannot be combined with ratio_model_zoo > 0: FSP / PFSP zoo opponents are "
                         "played without a partner")
    check_params_file(path)


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


def full_config(config: dict) -> dict:
    """default_config() updated with `config`, and the derived num_updates / num_minibatches"""
    cfg = dict(default_config())
    cfg.update(config)
    cfg["num_updates"] = cfg["total_timesteps"] // cfg["num_steps"] // cfg["num_envs"]   # ppo.py:225-227
    cfg["num_minibatches"] = cfg["num_envs"] * cfg["num_steps"] // cfg["minibatch_size"]  # ppo.py:228-230
    return cfg


class Learner:
    """One run's control plane of `train`: set-up, and per iteration the evaluations, opponent / zoo choice, rollout and
    GAE (`collect`), then logging and table rotation (`finish_iteration`) around an update step the caller runs -- alone
    (`train`) or grouped with other learners' (`train_population`)."""

    def __init__(self, config: dict, rng: int, tables: Optional[Sequence] = None, eval_table=None, device="cuda",
                 log_fn: Optional[Callable[[dict], None]] = None, eval_opp_params=None,
                 np_rng: Optional[np.random.Generator] = None, forward_pass_factory=None):
        make_fp = forward_pass_factory or make_forward_pass
        self.config = config = full_config(config)
        check_anchor_config(config)
        check_reward_mode(config)
        check_partner_config(config)
        self.log_fn = log_fn
        self.np_rng = np_rng or np.random.default_rng(config["seed"])
        self.dev = dev = torch.device(device)

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

        self.optimizer = make_optimizer(config)                                                       # ppo.py:195-211
        self.actor_forward_pass = make_fp(config["actor_activation"], config["actor_model_type"])
        rng, _rng = brandom.split(rng)
        params = init_params(_rng & 0x7FFFFFFF, dev)                                                  # ppo.py:240-243
        opt_state = self.optimizer.init(params)
        if config["load_initial_model"]:
            params = load_params(config["initial_model_path"], dev)                                   # ppo.py:246-248

        rng, self.eval_rng = brandom.split(rng)
        self.eval_env = eval_env = BridgeBidding(table=eval_table, device=dev)
        if eval_opp_params is None:
            eval_opp_params = (load_params(config["eval_opp_model_path"], dev) if config["eval_opp_model_path"]
                               else init_params(12345, dev))
        self.simple_evaluate, self.simple_duplicate_evaluate, self.duplicate_evaluate = make_evaluators(config, eval_env,
                                                                                                        eval_opp_params)

        opp_forward_pass = make_fp(config["opp_activation"], config["opp_model_type"])
        # the KL anchor: a fixed net of the actor's architecture, this learner's own (PBT's adopt keeps it)
        self.anchor_params, anchor_forward_pass = None, None
        if config["anchor_model_path"]:
            self.anchor_params = load_params(config["anchor_model_path"], dev)
            anchor_forward_pass = make_fp(config["actor_activation"], config["actor_model_type"])
        self.anchor_logits = None  # the latest roll-out's anchor logits [num_steps, num_envs, 38]
        # the fixed partner: a net of the actor's architecture, this learner's own (PBT's adopt keeps it), never trained
        self.partner_params, partner_forward_pass = None, None
        if config["partner_model_path"]:
            self.partner_params = load_params(config["partner_model_path"], dev)
            partner_forward_pass = make_fp(config["actor_activation"], config["actor_model_type"])
        self.envs = [BridgeBidding(table=t, device=dev) for t in tables]                              # ppo.py:296-303
        self.roll_outs = [make_roll_out(config, env, self.actor_forward_pass, opp_forward_pass, anchor_forward_pass,
                                        partner_forward_pass) for env in self.envs]
        self.calc_gae = make_calc_gae(config, self.actor_forward_pass)

        rng, _rng = brandom.split(rng)
        self.env, self.roll_out = self.envs[0], self.roll_outs[0]
        env_state = self.env.init(self.env.make_keys(_rng, config["num_envs"]))
        self.hash_index_list = np.arange(len(tables))
        self.steps, self.hash_index, self.board_count = 0, 0, 0
        terminated_count = torch.zeros((), dtype=torch.int64, device=dev)
        rng, _rng = brandom.split(rng)
        self.rng = rng
        self.runner_state = (params, opt_state, env_state, env_state.observation, terminated_count, _rng)

        if not config["self_play"]:
            self.opp_params = load_params(config["opp_model_path"], dev) if config["opp_model_path"] else eval_opp_params
        else:
            self.opp_params = params
        # past models.  ppo.py keeps them on disk (params-XXXXXXXX.pkl under save_model_path) and loads one at a time; here
        # they only exist when the league can use them.  They are a zoo.ModelZoo packed in HBM (allocated once for every save
        # the run makes, up to num_model_zoo): the PFSP probe is one league call and an opponent one device copy.  If that
        # pool does not fit in free device memory at the start (after the zoos of the learners set up before this one), or
        # when the opponent's forward is not the tensor-core one (which reads a packed opponent), they are host-memory NumPy
        # dicts (14.7 MB each), copied to the device one at a time and probed one match each.
        self.use_zoo = bool(config["self_play"]) and float(config["ratio_model_zoo"]) > 0.0
        zoo_capacity = min(config["num_model_zoo"], max(0, config["num_updates"] - 1) // config["save_model_interval"])
        self.zoo = []
        probe_envs = config["num_prioritized_envs"] if config["prioritized_fictitious"] else 0
        if self.use_zoo and isinstance(opp_forward_pass, ForwardPass) and device_zoo_fits(zoo_capacity, probe_envs, dev):
            self.zoo = ModelZoo(zoo_capacity, dev)
            if probe_envs:
                self.pfsp_probe = make_device_pfsp_probe(eval_env, config["actor_activation"], config["actor_model_type"],
                                                         probe_envs)
                self.pfsp_probe.reserve(self.zoo)             # all of the zoo's device memory is taken here, once
        self.device_zoo = isinstance(self.zoo, ModelZoo)
        self.save_dir = os.path.join(config["log_path"], config["exp_name"], config["save_model_path"])
        if config["save_model"]:
            os.makedirs(self.save_dir, exist_ok=True)
        self.logs = []
        self.pbt_lineage = None  # train_population with PBT: [iteration, parent, {key: value}] per PBT step

    def zoo_model(self, k: int):
        if self.device_zoo:
            return self.zoo.opponent(k)
        return {name: {kk: torch.as_tensor(v, device=self.dev) for kk, v in self.zoo[k][name].items()} for name in LAYERS}

    def collect(self, i: int):
        """Iteration i up to the update: saves, evaluations, opponent choice, rollout, GAE (ppo.py:351-477).  Returns
        (traj_batch, advantages, targets) for the update step of self.runner_state."""
        config, zoo, np_rng, eval_rng, dev = self.config, self.zoo, self.np_rng, self.eval_rng, self.dev
        runner_state = self.runner_state
        if i != 0 and i % config["save_model_interval"] == 0:                                      # ppo.py:351-362
            if self.device_zoo:
                zoo.append(runner_state[0])                  # keeps the newest zoo_capacity <= num_model_zoo models
            elif self.use_zoo:
                zoo.append(params_to_host(runner_state[0]))
                zoo[:] = zoo[-config["num_model_zoo"]:]
            if config["save_model"]:
                save_params(runner_state[0], os.path.join(self.save_dir, f"params-{i:08}.pkl"))
        t0 = time.time()
        partner = self.partner_params
        self.R = self.simple_evaluate(runner_state[0], eval_rng, partner_params=partner)          # ppo.py:365-368
        self.eval_log = {}
        if i % config["num_eval_step"] == 0:                                                      # ppo.py:369-374
            log_info, table_a_info, table_b_info = self.duplicate_evaluate(runner_state[0], eval_rng, partner_params=partner)
            self.eval_log = make_evaluate_log(log_info)
            if config["log_par"]:  # the same match against par: its initial state from the keys it was played from
                init_state = self.eval_env.init(self.duplicate_evaluate.buffers.keys)
                par = par_statistics(self.eval_env, init_state, table_a_info, table_b_info)
                self.eval_log.update({"eval/imp_vs_par": float(par["imp_vs_par"][0]),
                                      "eval/abs_imp_vs_par": float(par["abs_imp_vs_par"]),
                                      "eval/par_contract_rate": float(par["par_contract_rate"])})
        self.t_eval = time.time() - t0

        if config["self_play"]:                                                                   # ppo.py:376-470
            (imp_opp, _, _), _, _, _ = self.simple_duplicate_evaluate(runner_state[0], self.opp_params, eval_rng,
                                                                      team1_partner=partner)
            if imp_opp >= config["threshold_model_zoo"]:
                if len(zoo) != 0 and np_rng.binomial(1, config["ratio_model_zoo"]):
                    if config["prioritized_fictitious"]:
                        imp_list = np.zeros(len(zoo))
                        if self.device_zoo:  # the learner against every zoo model in one league call
                            imp_list[:] = [imp for imp, _, _ in self.pfsp_probe(runner_state[0], zoo, eval_rng)]
                        else:
                            for k in range(len(zoo)):  # one past model on the device at a time
                                (imp_list[k], _, _), _, _, _ = self.simple_duplicate_evaluate(runner_state[0], self.zoo_model(k),
                                                                                              eval_rng)
                        self.opp_params = self.zoo_model(int(np_rng.choice(len(zoo), p=pfsp_probabilities(imp_list,
                                                                                                           config["prior_t"]))))
                    else:
                        self.opp_params = self.zoo_model(int(np_rng.integers(len(zoo))))
                else:
                    self.opp_params = runner_state[0]
        (self.imp_opp_before, _, _), _, _, _ = self.simple_duplicate_evaluate(runner_state[0], self.opp_params, eval_rng,
                                                                              team1_partner=partner)
        torch.cuda.synchronize(dev)
        t1 = time.time()
        runner_state, traj_batch = self.roll_out(runner_state, self.opp_params, anchor_params=self.anchor_params,
                                                 partner_params=partner)                         # :472-475
        self.anchor_logits = self.roll_out.anchor_logits
        torch.cuda.synchronize(dev)
        t2 = time.time()
        advantages, targets = self.calc_gae(runner_state, traj_batch)                             # ppo.py:477
        torch.cuda.synchronize(dev)
        t3 = time.time()
        self.t_rollout, self.t_gae = t2 - t1, t3 - t2
        self.runner_state = runner_state
        return traj_batch, advantages, targets

    def update_kwargs(self) -> dict:
        """the update step's keywords for the latest roll-out: its anchor logits when this learner has an anchor"""
        return {} if self.anchor_params is None else {"anchor_logits": self.anchor_logits}

    def finish_iteration(self, i: int, runner_state, loss_info, t_update: float, emit: bool = True, anchor_kl=None) -> dict:
        """Iteration i after the update (ppo.py:479-549): the strength probe, the log, the table rotation.  `emit=False`
        leaves the log_fn call to the caller (`emit`), which adds entries to the log first.  `anchor_kl`: the update's
        per-minibatch KL to the anchor, [update_epochs, num_minibatches], logged as train/anchor_kl when there is an anchor."""
        config, dev = self.config, self.dev
        self.runner_state = runner_state
        (imp_opp_after, _, _), _, _, _ = self.simple_duplicate_evaluate(runner_state[0], self.opp_params, self.eval_rng,
                                                                        team1_partner=self.partner_params)
        self.steps += config["num_envs"] * config["num_steps"]
        total_loss, (value_loss, loss_actor, entropy, approx_kl, clipflacs, illegal_action_loss) = loss_info
        lr_now = self.optimizer.lr_at((i + 1) * config["update_epochs"] * config["num_minibatches"])
        board_num = int(runner_state[4])
        log = {                                                                                   # ppo.py:508-523
            "train/score": float(self.R), "train/total_loss": float(total_loss[-1][-1]),
            "train/value_loss": float(value_loss[-1][-1]), "train/loss_actor": float(loss_actor[-1][-1]),
            "train/illegal_action_loss": float(illegal_action_loss[-1][-1]), "train/policy_entropy": float(entropy[-1][-1]),
            "train/clipflacs": float(clipflacs[-1][-1]), "train/approx_kl": float(approx_kl[-1][-1]), "train/lr": lr_now,
            "train/imp_opp_before": float(self.imp_opp_before), "train/imp_opp_after": float(imp_opp_after),
            "board_num": board_num, "steps": self.steps,
            "time/eval": self.t_eval, "time/rollout": self.t_rollout, "time/calc_gae": self.t_gae, "time/update": t_update,
        }
        if self.anchor_params is not None:
            log["train/anchor_kl"] = float(anchor_kl[-1][-1])
        log.update(self.eval_log)
        self.logs.append(log)
        if emit:
            self.emit(log)
        if (board_num - self.board_count) // config["hash_size"] >= 1:                            # ppo.py:525-549
            self.hash_index += 1
            self.board_count = board_num
            if self.hash_index == len(self.hash_index_list):
                self.hash_index = 0
                self.np_rng.shuffle(self.hash_index_list)
            k = self.hash_index_list[self.hash_index]
            self.env, self.roll_out = self.envs[k], self.roll_outs[k]
            self.rng, _rng = brandom.split(self.rng)
            env_state = self.env.init(self.env.make_keys(_rng, config["num_envs"]))
            self.runner_state = (runner_state[0], runner_state[1], env_state, env_state.observation, runner_state[4], _rng)
            log["table"] = int(k)
        return log

    def emit(self, log: dict) -> None:
        if self.log_fn is not None:
            self.log_fn(log)

    def adopt(self, src: "Learner", values: dict) -> None:
        """PBT's exploit and explore: take `src`'s parameters and Adam state (device copies into this learner's own
        buffers, on the current stream) and set the config `values`, rebuilding the optimizer that captured them.  The
        update step holds the loss coefficients and optimizers and is the caller's to rebuild.  Env state, rollout key,
        table rotation, zoo, KL anchor, fixed partner and save directory stay this learner's; a self-play opponent becomes the new
        parameters."""
        params, opt_state = self.runner_state[:2]
        src_params, src_state = src.runner_state[:2]
        for name in LAYERS:
            for k in ("w", "b"):
                params[name][k].copy_(src_params[name][k])
        opt_state.mu.copy_(src_state.mu)
        opt_state.nu.copy_(src_state.nu)
        self.runner_state = (params, OptState(src_state.count, opt_state.mu, opt_state.nu)) + tuple(self.runner_state[2:])
        self.config.update(values)
        self.optimizer = make_optimizer(self.config)
        if self.config["self_play"]:
            self.opp_params = params

    def finish(self):
        """The final save (ppo.py:550-569); -> (runner_state, logs) as `train` returns them."""
        config = self.config
        if config["save_model"]:
            save_params(self.runner_state[0], os.path.join(self.save_dir, f"params-{config['num_updates']:08}.pkl"))
            with open(os.path.join(self.save_dir, f"opt_state-{config['num_updates']:08}.pkl"), "wb") as fh:
                st = self.runner_state[1]
                pickle.dump({"count": st.count, "mu": st.mu.cpu().numpy(), "nu": st.nu.cpu().numpy()}, fh)
            if self.pbt_lineage is not None:
                _pbt.write_lineage(os.path.join(self.save_dir, "pbt_lineage.json"), self.pbt_lineage)
        return self.runner_state, self.logs


def train(config: dict, rng: int, tables: Optional[Sequence] = None, eval_table=None, device="cuda",
          log_fn: Optional[Callable[[dict], None]] = None, eval_opp_params=None, np_rng: Optional[np.random.Generator] = None,
          forward_pass_factory=None, update_step_factory=None):
    """`forward_pass_factory(activation, model_type)` / `update_step_factory(config, forward_pass, optimizer)` replace
    `make_forward_pass` / `make_update_step` -- the hook the cuBLAS cross-check (scripts/torch_baseline.py) plugs into;
    the defaults are the tensor-core kernels and nothing else."""
    learner = Learner(config, rng, tables, eval_table, device, log_fn, eval_opp_params, np_rng, forward_pass_factory)
    update_step = (update_step_factory or make_update_step)(learner.config, learner.actor_forward_pass, learner.optimizer)
    for i in range(learner.config["num_updates"]):
        traj_batch, advantages, targets = learner.collect(i)
        t3 = time.time()
        runner_state, loss_info = update_step(learner.runner_state, traj_batch, advantages, targets,
                                              **learner.update_kwargs())                          # ppo.py:479-484
        torch.cuda.synchronize(learner.dev)
        learner.finish_iteration(i, runner_state, loss_info, time.time() - t3, anchor_kl=getattr(update_step, "anchor_kl", None))
    return learner.finish()


def train_population(configs: Sequence[dict], rngs: Sequence[int], tables: Optional[Sequence] = None, eval_table=None,
                     device="cuda", log_fns: Optional[Sequence[Optional[Callable[[dict], None]]]] = None,
                     eval_opp_params=None, np_rngs: Optional[Sequence[Optional[np.random.Generator]]] = None,
                     pbt: Optional[dict] = None):
    """`train` for K learners on one GPU.  Each learner runs its own control plane (evaluations, FSP / PFSP opponents and
    zoo, rollout, GAE, logging, table rotation) in turn, and the K updates of an iteration run as one grouped update step
    (update.make_population_update_step), so that the learners' GEMM tiles share the device.  configs[k] and rngs[k] give
    learner k exactly the run `train(configs[k], rngs[k], ...)` gives; the keys of update.POPULATION_SHARED_KEYS must be
    equal across learners (ValueError naming the first that is not).  -> [(runner_state, logs)] per learner.

    `pbt`: population-based training (brl_b200/pbt.py), a dict of options over default_pbt_config(): `interval`
    (iterations between rankings; 10), `metric` ("league": each learner's mean IMP in a round robin of the K current nets
    on `league_boards` (100) boards of the eval table; "score": its latest train/score), `quantile` (0.25: n = max(1,
    floor(quantile * K)) of the lowest learners each copy the parameters and Adam state of one of the n highest),
    `perturb_keys` (("lr", "ent_coef"): the winner's values the loser takes, each multiplied by a factor drawn from
    `perturb_factors`, (0.8, 1.25)) and `seed` (the population's generator of those draws).  Rankings run at iterations
    i > 0 with i % interval == 0, after every learner's finish_iteration; that iteration's logs gain pbt/fitness,
    pbt/rank (0 = fittest), pbt/parent (the learner copied, or -1) and pbt/<key> for each perturbed key before log_fns
    see them, and with save_model each learner's save directory gets a pbt_lineage.json.  ValueError (before any device work) for K < 2, a quantile outside (0, 0.5], a perturbed key that
    default_config() does not know or that the population shares, and the other bad options pbt.check_pbt_config lists.
    None (the default) trains the learners independently, as above.

    KL anchors: each learner has its own anchor net (anchor_model_path) and coefficient (anchor_kl_coef, which PBT may
    perturb); either every learner has an anchor or none has (ValueError naming anchor_model_path).

    Fixed partners: each learner has its own partner_model_path or none (the partner is not trained, so the grouped update
    is the same); every learner's partner is checked before any device work."""
    K = len(configs)
    if len(rngs) != K:
        raise ValueError("train_population needs one rng per config")
    full = [full_config(c) for c in configs]
    check_population_configs(full)
    for c in full:
        check_anchor_config(c)
        check_reward_mode(c)
        check_partner_config(c)
    anchored = [bool(c["anchor_model_path"]) for c in full]
    if any(anchored) and not all(anchored):
        raise ValueError(f"population learners must all have a KL anchor or none: anchor_model_path is set for learners "
                         f"{[k for k in range(K) if anchored[k]]} only")
    pbt_cfg = _pbt.check_pbt_config(pbt, K) if pbt is not None else None
    log_fns = list(log_fns) if log_fns is not None else [None] * K
    np_rngs = list(np_rngs) if np_rngs is not None else [None] * K
    learners = [Learner(configs[k], rngs[k], tables, eval_table, device, log_fns[k], eval_opp_params, np_rngs[k]) for k in range(K)]
    update_step = make_population_update_step([ln.config for ln in learners], learners[0].actor_forward_pass,
                                              [ln.optimizer for ln in learners])
    controller = _pbt.PopulationBasedTraining(pbt_cfg, learners) if pbt_cfg is not None else None
    dev = learners[0].dev
    for i in range(full[0]["num_updates"]):
        batches = [ln.collect(i) for ln in learners]
        t3 = time.time()
        anchor = {"anchor_logits": [ln.anchor_logits for ln in learners]} if any(anchored) else {}
        outs = update_step([ln.runner_state for ln in learners], [b[0] for b in batches], [b[1] for b in batches],
                           [b[2] for b in batches], **anchor)
        torch.cuda.synchronize(dev)
        t_update = time.time() - t3
        ranking = controller is not None and controller.due(i)
        anchor_kl = getattr(update_step, "anchor_kl", None) or [None] * K
        for k, (ln, (runner_state, loss_info)) in enumerate(zip(learners, outs)):
            ln.finish_iteration(i, runner_state, loss_info, t_update, emit=not ranking, anchor_kl=anchor_kl[k])
        if ranking:
            controller.step(i, learners)
            update_step = make_population_update_step([ln.config for ln in learners], learners[0].actor_forward_pass,
                                                      [ln.optimizer for ln in learners])
            for ln in learners:
                ln.emit(ln.logs[-1])
    return [ln.finish() for ln in learners]
