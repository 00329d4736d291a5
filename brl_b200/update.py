"""`make_update_step` of src/update.py:9-244: `update_epochs` passes over the rollout, each a
fresh permutation split into `num_minibatches` minibatches; per minibatch the net is re-run,
the PPO loss and its gradient are formed, and the optimizer steps.

One back end: `brl_ppo_grad` -- minibatch take, forward with kept activations, loss head + its backward, and the
backward GEMMs all in hand-written kernels on tcgen05 (csrc/brl_mlp_train.cu, three-term bf16 split = fp32-class
gradients) -- then `brl_mlp_adam_step` (clip + Adam + refresh of the kernels' weight layout in one pass).  No library
GEMM, no autograd tape.  (The cuBLAS-fp32 + autograd cross-check of this path is scripts/torch_baseline.py.)
Functional semantics are kept: the caller's `params` / `opt_state` are not modified (ppo.py
keeps the pre-update params as `opp_params`), a new flat copy is updated and returned.

KL anchor: `update_step(..., anchor_logits=)` with the roll-out's anchor logits [T, n, 38] adds config["anchor_kl_coef"] *
mean KL(policy || anchor) to every minibatch's loss (brl_ppo_grad_anchored); the per-minibatch KL, [update_epochs,
num_minibatches], is then `update_step.anchor_kl` after the call (None without an anchor)."""
from __future__ import annotations

import torch

from . import _lib, ops
from . import random as brandom
from .optim import OptState, flatten_params, update_mlp_grouped_
from .utils import WithOutputs

_STAT_NAMES = ("total_loss", "value_loss", "loss_actor", "entropy", "approx_kl", "clipflacs", "illegal_action_loss")


def _loss_settings(config, actor_forward_pass, who):
    """One learner's loss settings: (ppo_grad's flag keywords, its coefficient row [clip_eps, ent_coef, vf_coef,
    illegal_l2_coef], the illegal_action_loss statistic mode, brl_train_tune)."""
    flags = dict(value_clipping=bool(config.get("value_clipping", True)), reward_scaling=bool(config.get("reward_scaling", False)),
                 masked_policy=bool(config["actor_illegal_action_mask"]))
    coefs = [float(config["clip_eps"]), float(config["ent_coef"]), float(config["vf_coef"]),
             float(config.get("illegal_action_l2norm_coef", 0.0))]
    # illegal_action_loss = ||probs * ~mask||_2 / 2 is the SPECTRAL norm of the [minibatch, 38] matrix (src/update.py:141-142): a
    # 38 x 38 eigen-problem per minibatch.  With the default illegal_action_l2norm_coef = 0 it is a logged statistic only,
    # and ppo.py logs just the LAST minibatch of the last epoch (ppo.py:505, `illegal_action_loss[-1][-1]`).  "last" (default)
    # computes it for the last minibatch of every epoch and leaves NaN elsewhere in loss_info -- never a wrong number;
    # "all" fills every entry as the reference does, at ~19 us (11 %) per optimizer step (scripts/exp_gram_cost.py).
    # A non-zero coefficient needs the norm for the gradient and always computes it.
    stat_mode = config.get("illegal_action_loss_stat", "last")
    if stat_mode not in ("last", "all"):
        raise ValueError("illegal_action_loss_stat must be 'last' or 'all'")
    if getattr(actor_forward_pass, "precision", None) not in ("tc", "tc-bf16"):
        raise TypeError(f"{who} needs a brl_b200.models.ForwardPass (tensor-core ReLU net); there is no library back end on the "
                        "product path")
    return flags, coefs, stat_mode, int(config.get("brl_train_tune", 0))


def _flat_rollout(traj_batch, advantages, targets, batch_size):
    """The ppo_grad buffers of one learner's rollout, flat over (step, env) (src/update.py:195-197): obs, mask, action,
    old_log_prob, old_value, advantages, targets."""
    T, n = advantages.shape
    assert batch_size == T * n, "batch size must be equal to number of steps * number of envs"  # src/update.py:189-192
    obs = traj_batch.obs.reshape(batch_size, -1)
    if obs.dtype == torch.bool:
        obs = obs.view(torch.uint8)
    return (obs.contiguous(), traj_batch.legal_action_mask.reshape(batch_size, -1).view(torch.uint8).contiguous(),
            traj_batch.action.reshape(batch_size).contiguous(), traj_batch.log_prob.reshape(batch_size).contiguous(),
            traj_batch.value.reshape(batch_size).contiguous(), advantages.reshape(batch_size).contiguous(),
            targets.reshape(batch_size).contiguous())


def _flat_anchor(anchor_logits, batch_size):
    """the roll-out's anchor logits [T, n, 38] as the f32 [T * n, 38] rows of the flat rollout"""
    if anchor_logits.dtype != torch.float32 or anchor_logits.numel() != batch_size * ops.NUM_ACTIONS:
        raise ValueError("anchor_logits must be the roll-out's float32 [num_steps, num_envs, 38] anchor logits")
    return anchor_logits.reshape(batch_size, ops.NUM_ACTIONS).contiguous()


def _permutation(permutation_fn, rng, batch_size, device):
    """One epoch's minibatch order (src/update.py:193): `permutation_fn`, or torch.randperm seeded by the key."""
    if permutation_fn is not None:
        perm = permutation_fn(rng, batch_size)
    else:
        perm = torch.randperm(batch_size, generator=torch.Generator(device="cpu").manual_seed(rng & 0x7FFFFFFFFFFFFFFF))
    return perm.to(device=device, dtype=torch.int32).contiguous()


def _loss_info(stats):
    """loss_info from stats[update_epochs, num_minibatches, 8]: (total_loss, (value_loss, loss_actor, entropy, approx_kl,
    clipflacs, illegal_action_loss)), each [update_epochs, num_minibatches] (src/update.py:170-173, 226-229; read at
    ppo.py:487-506)"""
    cols = [stats[:, :, i] for i in range(7)]
    return cols[0], tuple(cols[1:])


def make_update_step(config, actor_forward_pass, optimizer, permutation_fn=None):
    """`permutation_fn(rng, batch_size) -> int64/32 tensor` replaces jax.random.permutation
    (src/update.py:193); default: torch.randperm seeded by the key (tests inject a fixed one)."""
    flags, coefs, stat_mode, tune = _loss_settings(config, actor_forward_pass, "make_update_step")
    cfg = dict(zip(("clip_eps", "ent_coef", "vf_coef", "illegal_l2_coef"), coefs), **flags)
    kl_coef = float(config.get("anchor_kl_coef", 0.0))
    out = {"anchor_kl": None}

    def update_step(runner_state, traj_batch, advantages, targets, anchor_logits=None):
        params, opt_state, env_state, last_obs, terminated_count, rng = runner_state
        dev = advantages.device
        nmb, mbs = int(config["num_minibatches"]), int(config["minibatch_size"])
        obs, mask, action, old_lp, old_v, adv, tgt = _flat_rollout(traj_batch, advantages, targets, nmb * mbs)
        anchor = {}
        if anchor_logits is not None:
            anchor = dict(anchor_logits=_flat_anchor(anchor_logits, nmb * mbs),
                          kl_coef=torch.tensor([kl_coef], dtype=torch.float32).to(dev))

        flat_p, new_params = flatten_params(params)
        if opt_state is None:
            opt_state = optimizer.init(params)
        state = OptState(opt_state.count, opt_state.mu.clone(), opt_state.nu.clone())
        n_epochs = int(config["update_epochs"])
        stats_all = torch.zeros((n_epochs, nmb, 8), dtype=torch.float32, device=dev)
        acc = ops.ppo_scratch(dev)
        blob = ops.mlp_pack_train(flat_p)
        scratch = ops.mlp_train_scratch(mbs, dev)
        flat_g = torch.empty_like(flat_p)
        for epoch in range(n_epochs):
            rng, _rng = brandom.split(rng)                                        # src/update.py:187
            perm = _permutation(permutation_fn, _rng, nmb * mbs, dev)
            for mb in range(nmb):                                                  # src/update.py:207-209
                ops.ppo_grad(obs, blob, scratch, perm[mb * mbs:(mb + 1) * mbs], mask, action, old_lp, old_v, adv, tgt,
                             flat_g, stats_all[epoch, mb], acc, tune=tune, illegal_stat=stat_mode == "all" or mb == nmb - 1,
                             **cfg, **anchor)                                      # src/update.py:164-167
                state = optimizer.update_mlp_(flat_p, flat_g, state, acc[14:15], blob)  # src/update.py:168-169
        out["anchor_kl"] = stats_all[:, :, 7] if anchor else None
        return (new_params, state, env_state, last_obs, terminated_count, rng), _loss_info(stats_all)

    return WithOutputs(update_step, out)


# Keys every learner of a population must share: they fix the shapes of the stacked buffers and the flags and tile widths
# of the grouped launches (brl_ppo_grad_grouped).  Everything else -- seed, lr, anneal_lr, the loss coefficients,
# max_grad_norm, gamma, gae_lambda, opponents -- may differ per learner.
POPULATION_SHARED_KEYS = ("num_envs", "num_steps", "minibatch_size", "update_epochs", "total_timesteps",
                          "actor_illegal_action_mask", "value_clipping", "reward_scaling", "global_gradient_clipping",
                          "illegal_action_loss_stat", "actor_model_type", "actor_activation", "brl_train_tune")


def check_population_configs(configs) -> None:
    """ValueError naming the first key of POPULATION_SHARED_KEYS on which two learners' configs differ."""
    if not configs:
        raise ValueError("a population needs at least one learner")
    _missing = object()
    for key in POPULATION_SHARED_KEYS:
        values = [c.get(key, _missing) for c in configs]
        if any(v != values[0] for v in values[1:]):
            raise ValueError(f"population learners must share config[{key!r}]; got {[None if v is _missing else v for v in values]}")


def make_population_update_step(configs, actor_forward_pass, optimizers, permutation_fn=None):
    """`make_update_step` for K learners whose optimizer steps run as one grouped step (ops.ppo_grad_grouped,
    optim.update_mlp_grouped_).  update_step(runner_states, traj_batches, advantages, targets) takes one entry per
    learner and returns K `(runner_state, loss_info)` pairs, each what `make_update_step(configs[k], ...)` returns for
    that learner: every learner draws its permutations from its own key, and its parameters, optimizer state and loss
    statistics are bit-identical to its solo update.  The stacked parameter, gradient, moment and blob buffers of the
    whole update are owned here; the returned params / opt_state are views into them.  `anchor_logits=`: one roll-out's
    anchor logits per learner (every learner has an anchor or none has); `update_step.anchor_kl` is then a list of each
    learner's [update_epochs, num_minibatches] KL."""
    configs = list(configs)
    check_population_configs(configs)
    if len(optimizers) != len(configs):
        raise ValueError("make_population_update_step needs one optimizer per config")
    if len(configs) > _lib.MAX_LEARNERS:
        raise ValueError(f"a population has at most {_lib.MAX_LEARNERS} learners")
    settings = [_loss_settings(c, actor_forward_pass, "make_population_update_step") for c in configs]
    flags, _, stat_mode, tune = settings[0]  # shared keys: equal for every learner
    coef_rows = [coefs for _, coefs, _, _ in settings]
    kl_coefs = [float(c.get("anchor_kl_coef", 0.0)) for c in configs]
    c0 = configs[0]
    K = len(configs)
    out = {"anchor_kl": None}

    def update_step(runner_states, traj_batches, advantages, targets, anchor_logits=None):
        if not (len(runner_states) == len(traj_batches) == len(advantages) == len(targets) == K):
            raise ValueError(f"update_step needs {K} runner states, trajectories, advantages and targets")
        if anchor_logits is not None:
            if len(anchor_logits) != K:
                raise ValueError(f"update_step needs {K} anchor logits")
            if any(a is None for a in anchor_logits):
                if all(a is None for a in anchor_logits):
                    anchor_logits = None
                else:
                    raise ValueError("population learners must all have a KL anchor (anchor_model_path) or none")
        dev = advantages[0].device
        nmb, mbs = int(c0["num_minibatches"]), int(c0["minibatch_size"])
        batch_size = nmb * mbs
        n_epochs = int(c0["update_epochs"])
        flat = [_flat_rollout(tb, adv, tgt, batch_size) for tb, adv, tgt in zip(traj_batches, advantages, targets)]
        obs_dtype = flat[0][0].dtype
        if any(f[0].dtype != obs_dtype for f in flat):
            raise ValueError("population learners must record observations of one dtype")

        n_params, blob_bytes = ops.mlp_num_params(), int(_lib.load().brl_mlp_train_blob_bytes())
        flat_p = torch.zeros((K, ops.mlp_param_stride()), dtype=torch.float32, device=dev)  # learner k: flat_p[k, :n_params]
        m = torch.zeros_like(flat_p)
        v = torch.zeros_like(flat_p)
        blob = torch.empty((K, blob_bytes), dtype=torch.uint8, device=dev)
        new_params, states, rngs, rest = [], [], [], []
        for k, (rs, opt) in enumerate(zip(runner_states, optimizers)):
            params, opt_state, env_state, last_obs, terminated_count, rng = rs
            _, p_k = flatten_params(params, out=flat_p[k, :n_params])
            if opt_state is None:
                opt_state = opt.init(params)
            m[k, :n_params].copy_(opt_state.mu)
            v[k, :n_params].copy_(opt_state.nu)
            ops.mlp_pack_train(flat_p[k, :n_params], out=blob[k])
            new_params.append(p_k)
            states.append(OptState(opt_state.count, m[k, :n_params], v[k, :n_params]))
            rngs.append(rng)
            rest.append((env_state, last_obs, terminated_count))
        flat_g = torch.zeros_like(flat_p)
        stats_all = torch.zeros((n_epochs, nmb, K, 8), dtype=torch.float32, device=dev)
        acc = torch.zeros((K, _lib.PPO_SCRATCH_BYTES // 8), dtype=torch.float64, device=dev)
        scratch = torch.empty(ops.ppo_grad_grouped_scratch_bytes(K, mbs), dtype=torch.uint8, device=dev)
        coefs = torch.tensor(coef_rows, dtype=torch.float32).to(dev)
        anchor = {}
        if anchor_logits is not None:
            flat_anchor = [_flat_anchor(a, batch_size) for a in anchor_logits]  # alive until the update returns
            anchor = dict(anchor_logits=torch.tensor([a.data_ptr() for a in flat_anchor], dtype=torch.int64).to(dev),
                          kl_coef=torch.tensor(kl_coefs, dtype=torch.float32).to(dev))

        for epoch in range(n_epochs):
            perms = []
            for k in range(K):
                rngs[k], _rng = brandom.split(rngs[k])                            # src/update.py:187
                perms.append(_permutation(permutation_fn, _rng, batch_size, dev))
            # this epoch's trajectory tables, one [K, 8] per minibatch: the index column steps through each permutation
            base = torch.tensor([ops.ppo_trajectory_row(f[0], perms[k], *f[1:]) for k, f in enumerate(flat)], dtype=torch.int64)
            tables = base.repeat(nmb, 1, 1)
            tables[:, :, 1] += torch.arange(nmb, dtype=torch.int64)[:, None] * (4 * mbs)  # int32 index: 4 bytes a row
            tables = tables.pin_memory().to(dev, non_blocking=True)
            for mb in range(nmb):
                ops.ppo_grad_grouped(tables[mb], coefs, blob, scratch, flat_g, stats_all[epoch, mb], acc, batch=mbs,
                                     obs_dtype=obs_dtype, illegal_stat=stat_mode == "all" or mb == nmb - 1, tune=tune, **flags,
                                     **anchor)
                states = update_mlp_grouped_(optimizers, flat_p, flat_g, m, v, states, acc, blob)

        results = []
        for k in range(K):
            env_state, last_obs, terminated_count = rest[k]
            results.append(((new_params[k], states[k], env_state, last_obs, terminated_count, rngs[k]), _loss_info(stats_all[:, :, k])))
        out["anchor_kl"] = [stats_all[:, :, k, 7] for k in range(K)] if anchor else None
        return results

    return WithOutputs(update_step, out)
