"""Env wrappers of src/utils.py: `auto_reset` and the four-call "quad" steps.

Same names, argument meaning and results as the reference; the difference is that the
env is natively batched and the wrappers map onto kernel flags instead of traced
`lax.cond`s (which, under vmap, execute `env.init` for every env on every sub-step):
  auto_reset               -> brl_step with BRL_F_AUTORESET      (src/utils.py:9-58)
  rewards1+..+4, OR of terminated -> BRL_F_ACCUMULATE / BRL_F_QUAD_LAST (src/utils.py:126-128)
"""
from __future__ import annotations

import torch

from . import ops
from . import random as brandom
from .env import BridgeBidding, State


class WithOutputs:
    """A callable plus outputs it leaves beside its return value, read as attributes (`roll_out.anchor_logits`,
    `update_step.anchor_kl`): `fn` writes them into the dict `out`.  The function does not refer to the object that
    exposes them, so a roll-out or update step is freed by reference counting when its last user drops it -- a reference
    cycle would leave its CUDA graphs to the garbage collector, which may run inside another graph's capture."""
    __slots__ = ("_fn", "_out")

    def __init__(self, fn, out: dict):
        self._fn, self._out = fn, out

    def __call__(self, *args, **kwargs):
        return self._fn(*args, **kwargs)

    def __getattr__(self, name):
        try:
            return self._out[name]
        except KeyError:
            raise AttributeError(name) from None


class _AutoResetStep:
    def __init__(self, env: BridgeBidding):
        self.env = env

    def __call__(self, state: State, action: torch.Tensor) -> State:
        return self.env.step(state, action, autoreset=True)


def auto_reset(step_fn, init_fn):
    """src/utils.py:9-58.  `step_fn`/`init_fn` must be `env.step`/`env.init` of one env."""
    env = getattr(step_fn, "__self__", None)
    if not isinstance(env, BridgeBidding) or getattr(init_fn, "__self__", None) is not env:
        raise TypeError("auto_reset(step_fn, init_fn) expects env.step and env.init of a brl_b200.BridgeBidding")
    return _AutoResetStep(env)


def _env_of(step_fn):
    if isinstance(step_fn, _AutoResetStep):
        return step_fn.env, True
    env = getattr(step_fn, "__self__", None)
    if isinstance(env, BridgeBidding):
        return env, False
    raise TypeError("step_fn must be env.step or auto_reset(env.step, env.init)")


class _QuadStep:
    """Four consecutive env sub-steps (src/utils.py:69-128): the given action, then opp /
    actor / opp nets act on the fresh observation; returns the last state with
    rewards = sum of the four and terminated = OR of the four.

    Sub-step 3 is the partner's slot.  Given `partner_forward_pass` / `partner_params`, that net acts there instead of the
    actor (still sampled in "sample" mode, and still no recorded transition).  The slot is positional, as in the reference:
    after an auto-reset inside the quad step the seat to act at sub-step 3 may belong to the other team, and the partner's
    net then acts for that team, as the actor's would without a partner."""

    def __init__(self, step_fn, actor_forward_pass, actor_params, opp_forward_pass, opp_params, mode: str,
                 partner_forward_pass=None, partner_params=None):
        self.env, self.autoreset = _env_of(step_fn)
        self.actor_fp, self.actor_params = actor_forward_pass, actor_params
        self.opp_fp, self.opp_params = opp_forward_pass, opp_params
        if (partner_forward_pass is None) != (partner_params is None):
            raise ValueError("a partner needs both partner_forward_pass and partner_params")
        self.partner_fp, self.partner_params = (partner_forward_pass, partner_params) if partner_params is not None else \
            (actor_forward_pass, actor_params)
        self.mode = mode  # "sample" | "deterministic" | "free-run"
        self._scratch = None
        self._mid_obs = None
        self.trace = None  # tests set a list here to receive the four sub-step action tensors

    def _buffers(self, n, device):
        if self._scratch is None or self._scratch[0].shape[0] != n:
            self._scratch = (torch.empty(n, dtype=torch.int32, device=device),)
        return self._scratch

    def _policy_action(self, fp, params, state: State, seed: int, sample: bool, act_buf):
        fp.act(params, state.observation, state._mask_u8, act_buf, sample=sample, seed=seed, env_offset=self.env.env_offset)
        return act_buf

    def __call__(self, state: State, action: torch.Tensor, rng: int, *, out_state: State = None) -> State:
        env = self.env
        n = state.num_envs
        (act_buf,) = self._buffers(n, env.device)
        # sub-step 1 writes fresh rewards/terminated, sub-steps 2-4 accumulate into them
        packed, out = (out_state._packed, out_state.outputs()) if out_state is not None else env._fresh(n)
        kw = dict(autoreset=self.autoreset, illegal_penalty=env.illegal_penalty, illegal_bonus=env.illegal_bonus)
        # the observations of sub-steps 1-3 are read by a policy net only (the caller sees the 4th): when the nets
        # take bf16 input, write those straight in bf16 into a private buffer (no cast launch, half the bytes)
        mid = out
        if self.mode != "free-run" and getattr(self.actor_fp, "input_dtype", None) == torch.bfloat16 and \
                getattr(self.opp_fp, "input_dtype", None) == torch.bfloat16 and \
                getattr(self.partner_fp, "input_dtype", None) == torch.bfloat16 and out.observation.dtype != torch.bfloat16:
            if self._mid_obs is None or self._mid_obs.shape[0] != n:
                self._mid_obs = torch.empty((n, ops.OBS_DIM), dtype=torch.bfloat16, device=env.device)
            mid = State(env, packed, out).outputs()
            mid.observation = self._mid_obs
        ops.step(state._packed, action.to(torch.int32), env.table, packed, mid, **kw)
        if self.trace is not None:
            self.trace.append(action.clone())
        cur = State(env, packed, mid)
        plan = ((self.opp_fp, self.opp_params), (self.partner_fp, self.partner_params), (self.opp_fp, self.opp_params))
        for k, (fp, params) in enumerate(plan):
            rng, sub = brandom.split(rng)
            if self.mode == "free-run" and k != 1:
                act_buf.zero_()  # opponents always pass (src/utils.py:217,235)
            else:
                sample = self.mode == "sample"
                self._policy_action(fp, params, cur, sub, sample, act_buf)
            if self.trace is not None:
                self.trace.append(act_buf.clone())
            ops.step(packed, act_buf, env.table, packed, out if k == 2 else mid, accumulate=True, quad_last=(k == 2), **kw)
        return State(env, packed, out)


def single_play_step_two_policy_commpetitive(step_fn, actor_forward_pass, actor_params, opp_forward_pass, opp_params,
                                             partner_forward_pass=None, partner_params=None):
    """src/utils.py:61-130 (sampled opponents / partner); the partner is the actor unless given"""
    return _QuadStep(step_fn, actor_forward_pass, actor_params, opp_forward_pass, opp_params, "sample",
                     partner_forward_pass, partner_params)


def single_play_step_two_policy_commpetitive_deterministic(step_fn, actor_forward_pass, actor_params,
                                                           opp_forward_pass, opp_params, partner_forward_pass=None,
                                                           partner_params=None):
    """src/utils.py:133-202 (argmax opponents / partner); the partner is the actor unless given"""
    return _QuadStep(step_fn, actor_forward_pass, actor_params, opp_forward_pass, opp_params, "deterministic",
                     partner_forward_pass, partner_params)


def single_play_step_free_run(step_fn, actor_forward_pass, actor_params, opp_forward_pass, opp_params,
                              partner_forward_pass=None, partner_params=None):
    """src/utils.py:205-246 (opponents always pass, partner argmax); the partner is the actor unless given"""
    return _QuadStep(step_fn, actor_forward_pass, actor_params, opp_forward_pass, opp_params, "free-run",
                     partner_forward_pass, partner_params)


def normal_step(step_fn):
    """src/utils.py:249-254"""
    def wrapped_step_fn(state, action, rng):
        return step_fn(state, action)
    return wrapped_step_fn
