"""Torch-tensor front-end of the stream-first C-ABI ops (include/brl_b200.h).

PyTorch is plumbing here: it owns device memory and the current CUDA stream; all
arithmetic happens in the hand-written sm_100a kernels behind `_lib.call`.
Every function enqueues on `torch.cuda.current_stream()` and never synchronises.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from ._lib import (BrlParams, F_ACCUMULATE, F_AUTORESET, F_MLP_BF16, F_OBS_BF16, F_OBS_U8, F_QUAD_LAST,
                   F_RANDOM_ACTION, F_RESULT_I16, F_SAMPLE, F_UNIFORM_U16)

NUM_ACTIONS = 38
OBS_DIM = 480
STATE_PLANES = 5

_OBS_FLAG = {torch.float32: 0, torch.uint8: F_OBS_U8, torch.bool: F_OBS_U8, torch.bfloat16: F_OBS_BF16}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.BrlError("brl_b200 ops need CUDA tensors (there is no CPU path)")
    if not t.is_contiguous():
        raise _lib.BrlError("brl_b200 ops need contiguous tensors")
    return t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _call(name: str, buffers, params) -> None:
    # buffers were validated (CUDA, contiguous) while the list was built; only then touch the stream
    _lib.call(name, _stream(), buffers, params)


def _params(n, *, flags=0, env_offset=0, stride=0, seed=0, n_deals=0, step=0, k_steps=0, illegal_penalty=-1.0,
            illegal_bonus=1.0, gamma=0.0, gae_lambda=0.0) -> BrlParams:
    return BrlParams(int(n), int(env_offset), int(stride or n), int(seed) & 0xFFFFFFFFFFFFFFFF, int(n_deals), int(flags),
                     int(step) & 0xFFFFFFFF, int(k_steps), float(illegal_penalty), float(illegal_bonus), float(gamma),
                     float(gae_lambda))


def obs_flag(dtype: torch.dtype) -> int:
    try:
        return _OBS_FLAG[dtype]
    except KeyError:
        raise _lib.BrlError(f"observation dtype {dtype} not supported (float32, uint8/bool, bfloat16)") from None


def new_state(n: int, device) -> torch.Tensor:
    """Packed env state: uint4[5][n] plane-major, seen from torch as int32[5, n, 4]."""
    return torch.empty((STATE_PLANES, n, 4), dtype=torch.int32, device=device)


def _trajectory(shape, dtype: torch.dtype, device) -> torch.Tensor:
    """Uninitialised tensor in compressible device memory (brl_alloc_compressible); freed with its last view."""
    nbytes = dtype.itemsize
    for d in shape:
        nbytes *= d
    if nbytes == 0:
        return torch.empty(shape, dtype=dtype, device=device)
    device = torch.device(device)
    index = device.index if device.index is not None else torch.cuda.current_device()
    buf = _lib.CompressibleBuffer(nbytes, index)
    return torch.as_tensor(buf, device=torch.device("cuda", index)).view(dtype).view(shape)


class EnvOutputs:
    """The Env surface brl consumes (src/roll_out.py:72-100): caller-owned output buffers.

    With rows > 0 the observation and mask trajectories ([rows, n, ...], almost all zero bytes) live in compressible
    device memory, which shrinks their write-back to DRAM; the per-step outputs (rows = 0) come from torch."""

    __slots__ = ("observation", "legal_action_mask", "rewards", "terminated", "current_player")

    def __init__(self, n: int, device, obs_dtype=torch.float32, rows: int = 0):
        lead = (rows, n) if rows else (n,)
        odt = torch.uint8 if obs_dtype == torch.bool else obs_dtype
        if rows:
            self.observation = _trajectory(lead + (OBS_DIM,), odt, device)
            self.legal_action_mask = _trajectory(lead + (NUM_ACTIONS,), torch.uint8, device)
        else:
            self.observation = torch.empty(lead + (OBS_DIM,), dtype=odt, device=device)
            self.legal_action_mask = torch.empty(lead + (NUM_ACTIONS,), dtype=torch.uint8, device=device)
        self.rewards = torch.empty(lead + (4,), dtype=torch.float32, device=device)
        self.terminated = torch.empty(lead, dtype=torch.uint8, device=device)
        self.current_player = torch.empty(lead, dtype=torch.int8, device=device)

    def ptrs(self):
        return [_ptr(self.observation), _ptr(self.legal_action_mask), _ptr(self.rewards), _ptr(self.terminated),
                _ptr(self.current_player)]

    def flag(self) -> int:
        return obs_flag(self.observation.dtype)


def make_keys(seed: int, n: int, device, env_offset: int = 0) -> torch.Tensor:
    keys = torch.empty(n, dtype=torch.int64, device=device)
    _call("brl_make_keys", [_ptr(keys)], _params(n, seed=seed, env_offset=env_offset))
    return keys


def init(keys: torch.Tensor, table: torch.Tensor, state: torch.Tensor, out: EnvOutputs, tune: int = 0) -> None:
    n = keys.shape[0]
    _call("brl_init", [_ptr(keys), _ptr(table), _ptr(state), *out.ptrs()],
              _params(n, n_deals=table.shape[0], stride=state.shape[1], flags=out.flag() | tune))


def reset_fields(deal, dealer, vul_ns, vul_ew, players, rng_key, table, state, out: EnvOutputs) -> None:
    n = deal.shape[0]
    _call("brl_reset_fields", [_ptr(deal), _ptr(dealer), _ptr(vul_ns), _ptr(vul_ew), _ptr(players), _ptr(rng_key), _ptr(table),
               _ptr(state), *out.ptrs()],
              _params(n, n_deals=table.shape[0], stride=state.shape[1], flags=out.flag()))


def step(state_in, action, table, state_out, out: EnvOutputs, *, autoreset=False, random_action=False,
         accumulate=False, quad_last=False, seed=0, step_index=0, env_offset=0, action_out=None,
         illegal_penalty=-1.0, illegal_bonus=1.0, tune: int = 0) -> None:
    n = state_in.shape[1]
    flags = out.flag() | tune
    flags |= F_AUTORESET if autoreset else 0
    flags |= F_RANDOM_ACTION if random_action else 0
    flags |= F_ACCUMULATE if accumulate else 0
    flags |= F_QUAD_LAST if quad_last else 0
    _call("brl_step", [_ptr(state_in), _ptr(action), _ptr(table), _ptr(state_out), *out.ptrs(), _ptr(action_out)],
              _params(n, flags=flags, n_deals=table.shape[0], stride=state_in.shape[1], seed=seed, step=step_index,
                      env_offset=env_offset, illegal_penalty=illegal_penalty, illegal_bonus=illegal_bonus))


class TableInfoBuffers:
    """src/duplicate.py:138-144 Table_info as SoA device buffers."""

    __slots__ = ("terminated", "rewards", "last_bid", "last_bidder", "call_x", "call_xx")

    def __init__(self, n: int, device):
        self.terminated = torch.zeros(n, dtype=torch.uint8, device=device)
        self.rewards = torch.zeros((n, 4), dtype=torch.float32, device=device)
        self.last_bid = torch.full((n,), -1, dtype=torch.int32, device=device)
        self.last_bidder = torch.full((n,), -1, dtype=torch.int32, device=device)
        self.call_x = torch.zeros(n, dtype=torch.uint8, device=device)
        self.call_xx = torch.zeros(n, dtype=torch.uint8, device=device)

    def ptrs(self):
        return [_ptr(getattr(self, k)) for k in self.__slots__]


def duplicate_step(state_in, action, table, info_a: TableInfoBuffers, info_b: TableInfoBuffers, state_out,
                   out: EnvOutputs, illegal_penalty=-1.0, illegal_bonus=1.0) -> None:
    n = state_in.shape[1]
    _call("brl_duplicate_step", [_ptr(state_in), _ptr(action), _ptr(table), *info_a.ptrs(), *info_b.ptrs(), _ptr(state_out), *out.ptrs()],
              _params(n, flags=out.flag(), n_deals=table.shape[0], stride=state_in.shape[1],
                      illegal_penalty=illegal_penalty, illegal_bonus=illegal_bonus))


def duplicate_init(state_in, table, state_out, out: EnvOutputs) -> None:
    n = state_in.shape[1]
    _call("brl_duplicate_init", [_ptr(state_in), _ptr(table), _ptr(state_out), *out.ptrs()],
              _params(n, flags=out.flag(), n_deals=table.shape[0], stride=state_in.shape[1]))


def observe(state, table, obs: torch.Tensor, player_id: Optional[torch.Tensor] = None, tune: int = 0) -> None:
    n = state.shape[1]
    _call("brl_observe", [_ptr(state), _ptr(player_id), _ptr(table), _ptr(obs)],
              _params(n, flags=obs_flag(obs.dtype) | tune, n_deals=table.shape[0], stride=state.shape[1]))


def legal_mask(state, mask: torch.Tensor, tune: int = 0) -> None:
    n = state.shape[1]
    _call("brl_legal_mask", [_ptr(state), _ptr(mask)], _params(n, stride=state.shape[1], flags=tune))


def rollout_random(state, table, k_steps: int, out: Optional[EnvOutputs], *, seed=0, step0=0, env_offset=0,
                   action_out=None, stats=None, obs_only: Optional[torch.Tensor] = None, tune: int = 0,
                   uniforms: Optional[torch.Tensor] = None, result16: Optional[torch.Tensor] = None) -> None:
    """K auto-reset random-legal steps in ONE launch; `out` holds [K, n, ...] trajectories.
    `uniforms`: caller-owned randomness, int32/uint32 [K, n], or int16/uint16 [K, n] (stands for u16 << 16);
    `result16`: int16 [K, n] compact result = 2 * rewards[player 0] + terminated (decode_result16)."""
    n = state.shape[1]
    extra = 0
    if uniforms is not None and uniforms.element_size() == 2:
        extra |= F_UNIFORM_U16
    if result16 is not None:
        if result16.dtype != torch.int16:
            raise TypeError("result16 must be an int16 tensor")
        extra |= F_RESULT_I16
    if out is not None:
        ptrs, flag = out.ptrs(), out.flag()
    else:
        ptrs = [_ptr(obs_only), None, None, None, None]
        flag = obs_flag(obs_only.dtype) if obs_only is not None else 0
    _call("brl_rollout_random", [_ptr(state), _ptr(table), *ptrs, _ptr(action_out), _ptr(stats), _ptr(uniforms),
                                 _ptr(result16)],
              _params(n, flags=flag | tune | extra, n_deals=table.shape[0], stride=state.shape[1], seed=seed, step=step0,
                      env_offset=env_offset, k_steps=k_steps))


def decode_result16(result16: torch.Tensor):
    """compact rollout result -> (rewards f32[..., 4], terminated u8[...]) exactly as the Env surface gives them"""
    w = result16.to(torch.int32)
    s = (w >> 1).to(torch.float32)
    return torch.stack((s, s, -s, -s), dim=-1), (w & 1).to(torch.uint8)


def imp_reward(a_rewards, b_rewards, out) -> None:
    _call("brl_imp_reward", [_ptr(a_rewards), _ptr(b_rewards), _ptr(out)], _params(a_rewards.shape[0]))


def gae(done, value, reward, last_val, adv, targets, gamma: float, gae_lambda: float) -> None:
    t, n = done.shape
    _call("brl_gae", [_ptr(done), _ptr(value), _ptr(reward), _ptr(last_val), _ptr(adv), _ptr(targets)],
              _params(n, k_steps=t, gamma=gamma, gae_lambda=gae_lambda))


def categorical(logits, mask, action, log_prob, *, sample=False, seed=0, env_offset=0, step_index=0) -> None:
    n = logits.shape[0]
    _call("brl_categorical", [_ptr(logits), _ptr(mask), _ptr(action), _ptr(log_prob)],
              _params(n, flags=F_SAMPLE if sample else 0, seed=seed, env_offset=env_offset, step=step_index))


def match_stats(x: torch.Tensor, sums: torch.Tensor) -> None:
    _call("brl_match_stats", [_ptr(x), _ptr(sums)], _params(x.shape[0]))


def gather_reward(rewards, actor, out, scale: float, done: Optional[torch.Tensor] = None,
                  count: Optional[torch.Tensor] = None) -> None:
    """reward = rewards[actor] / scale (src/roll_out.py:86-94); with `done` (u8) and `count` (int64[1]): count += sum(done)
    in the same launch (src/roll_out.py:85)."""
    counting = done is not None and count is not None
    _call("brl_gather_reward", [_ptr(rewards), _ptr(actor), _ptr(out), _ptr(done) if counting else None,
                                _ptr(count) if counting else None],
          _params(rewards.shape[0], gamma=scale, flags=_lib.F_COUNT_DONE if counting else 0))


def par(state_packed, table, out, contract: Optional[torch.Tensor] = None) -> None:
    """Double-dummy par of each env's board (DESIGN.md f13): `out` f32[n, 4] in the rewards layout, by player id
    (p, p, -p, -p) with p the par of the team of player ids {0, 1}; `contract` i32[n]: -1 when passed out, else
    bid | declarer_seat << 8 | doubled << 10."""
    n = state_packed.shape[1]
    _call("brl_par", [_ptr(state_packed), _ptr(table), _ptr(out), _ptr(contract)],
          _params(n, stride=state_packed.shape[1], n_deals=table.shape[0]))


def par_stats(state_packed, table, rewards_a, last_bid_a, last_bidder_a, rewards_b, last_bid_b, last_bidder_b,
              sums: torch.Tensor) -> None:
    """sums f64[8] += {tables, sum IMP vs par, sum IMP^2, sum |IMP|, #par contract reached} of a duplicate match for the team
    of player ids {0, 1}; `state_packed` is table A's initial state, the rest the two tables' Table_info fields."""
    n = state_packed.shape[1]
    _call("brl_par_stats", [_ptr(state_packed), _ptr(table), _ptr(rewards_a), _ptr(last_bid_a), _ptr(last_bidder_a),
                            _ptr(rewards_b), _ptr(last_bid_b), _ptr(last_bidder_b), _ptr(sums)],
          _params(n, stride=state_packed.shape[1], n_deals=table.shape[0]))


def gather_reward_par(rewards, actor, par, done, out, count: Optional[torch.Tensor] = None) -> None:
    """reward = done ? IMP(rewards[actor] - par[actor]) / 24 : 0, with `par` from `par` on the state before the step;
    with `count` (int64[1]): count += sum(done) in the same launch."""
    _call("brl_gather_reward_par", [_ptr(rewards), _ptr(actor), _ptr(par), _ptr(done), _ptr(out), _ptr(count)],
          _params(rewards.shape[0], flags=_lib.F_COUNT_DONE if count is not None else 0))


def mlp_pack(weights, biases, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Six haiku-layout fp32 (w[in,out], b[out]) pairs -> the packed bf16 hi/lo parameter blob (`out`: re-pack in place)."""
    dev = weights[0].device
    blob = out if out is not None else torch.empty(_lib.load().brl_mlp_packed_bytes(), dtype=torch.uint8, device=dev)
    ws = [w.detach().to(torch.float32).contiguous() for w in weights]
    bs = [b.detach().to(torch.float32).contiguous() for b in biases]
    _call("brl_mlp_pack", [_ptr(t) for t in ws] + [_ptr(t) for t in bs] + [_ptr(blob)], _params(0))
    return blob


def obs_to_bf16(obs: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """0/1 observation in a reference dtype (f32 / u8 / bool) -> bf16 for the tensor-core forward."""
    if obs.dtype == torch.bfloat16:
        return obs
    n = obs.shape[0]
    if out is None:
        out = torch.empty((n, OBS_DIM), dtype=torch.bfloat16, device=obs.device)
    src = obs.view(torch.uint8) if obs.dtype == torch.bool else obs
    if src.dtype not in (torch.float32, torch.uint8):
        raise _lib.BrlError(f"observation dtype {obs.dtype} not supported")
    _call("brl_obs_to_bf16", [_ptr(src), _ptr(out)], _params(n, flags=F_OBS_U8 if src.dtype == torch.uint8 else 0))
    return out


def mlp_scratch(n: int, device) -> torch.Tensor:
    return torch.empty(_lib.load().brl_mlp_scratch_bytes(n), dtype=torch.uint8, device=device)


def mlp_forward(obs_bf16: torch.Tensor, packed: torch.Tensor, scratch: torch.Tensor, logits: torch.Tensor,
                value: torch.Tensor, single_bf16: bool = False, tune: int = 0) -> None:
    """logits f32[n,38], value f32[n] = DeepMind MLP(obs) on tcgen05 (3-term bf16 split unless single_bf16)."""
    n = obs_bf16.shape[0]
    if obs_bf16.dtype != torch.bfloat16:
        raise _lib.BrlError("mlp_forward needs a bf16 observation (ops.obs_to_bf16)")
    if scratch.numel() < _lib.load().brl_mlp_scratch_bytes(n):
        raise _lib.BrlError("mlp_forward: scratch too small (ops.mlp_scratch)")
    _call("brl_mlp_forward", [_ptr(obs_bf16), _ptr(packed), _ptr(scratch), _ptr(logits), _ptr(value)],
          _params(n, flags=(F_MLP_BF16 if single_bf16 else 0) | tune))


def policy_act(obs_bf16: torch.Tensor, packed: torch.Tensor, scratch: torch.Tensor, mask: Optional[torch.Tensor],
               action: torch.Tensor, log_prob: Optional[torch.Tensor] = None, value: Optional[torch.Tensor] = None,
               logits: Optional[torch.Tensor] = None, *, sample: bool = False, seed: int = 0, env_offset: int = 0,
               step_index: int = 0, single_bf16: bool = False, tune: int = 0, seed_salt: Optional[torch.Tensor] = None) -> None:
    """forward.apply + masked Categorical sample / mode (+ log_prob, value, logits on request) in one call
    (src/roll_out.py:73-81); same noise stream as `categorical`, so it equals mlp_forward followed by categorical."""
    n = obs_bf16.shape[0]
    if obs_bf16.dtype != torch.bfloat16:
        raise _lib.BrlError("policy_act needs a bf16 observation (ops.obs_to_bf16)")
    if scratch.numel() < _lib.load().brl_mlp_scratch_bytes(n):
        raise _lib.BrlError("policy_act: scratch too small (ops.mlp_scratch)")
    _call("brl_policy_act", [_ptr(obs_bf16), _ptr(packed), _ptr(scratch), _ptr(mask), _ptr(action), _ptr(log_prob), _ptr(value),
                             _ptr(logits), _ptr(seed_salt)],
          _params(n, flags=(F_MLP_BF16 if single_bf16 else 0) | (F_SAMPLE if sample else 0) | tune |
                  (_lib.F_SEED_SALT if seed_salt is not None else 0), seed=seed,
                  env_offset=env_offset, step=step_index))


def mlp_rows_scratch(n_rows: int, device) -> torch.Tensor:
    return torch.empty(_lib.load().brl_mlp_rows_scratch_bytes(n_rows), dtype=torch.uint8, device=device)


def policy_act_rows(obs_bf16: torch.Tensor, packed: torch.Tensor, scratch: torch.Tensor, mask: Optional[torch.Tensor],
                    action: torch.Tensor, rows: torch.Tensor, log_prob: Optional[torch.Tensor] = None,
                    logits: Optional[torch.Tensor] = None, *, sample: bool = False,
                    seed: int = 0, env_offset: int = 0, step_index: int = 0, single_bf16: bool = False, tune: int = 0) -> None:
    """`policy_act` restricted to the envs listed in `rows` (int32): only their observations are read and only their
    action / log_prob entries written (src/evaluation.py:124-151 without forwarding envs a net does not decide)."""
    n = rows.shape[0]
    if n == 0:
        return
    if obs_bf16.dtype != torch.bfloat16 or rows.dtype != torch.int32:
        raise _lib.BrlError("policy_act_rows needs a bf16 observation and int32 rows")
    if scratch.numel() < _lib.load().brl_mlp_rows_scratch_bytes(n):
        raise _lib.BrlError("policy_act_rows: scratch too small (ops.mlp_rows_scratch)")
    _call("brl_policy_act_rows", [_ptr(obs_bf16), _ptr(packed), _ptr(scratch), _ptr(mask), _ptr(action), _ptr(rows), _ptr(log_prob),
                                  _ptr(logits)],
          _params(n, flags=(F_MLP_BF16 if single_bf16 else 0) | (F_SAMPLE if sample else 0) | tune, seed=seed,
                  env_offset=env_offset, step=step_index))


def team_rows(current_player: torch.Tensor, done: Optional[torch.Tensor], rows1: torch.Tensor, rows2: torch.Tensor,
              counts: torch.Tensor) -> None:
    """rows of the live envs (done == 0) split by acting team: players 0/1 -> rows1, players 2/3 -> rows2; counts i32[2]."""
    _call("brl_team_rows", [_ptr(current_player), _ptr(done), _ptr(rows1), _ptr(rows2), _ptr(counts)],
          _params(current_player.shape[0]))


def ppo_scratch(device) -> torch.Tensor:
    """scratch of ppo_loss / ppo_grad as a float64 tensor (element 14 = sum of squares of the gradient after ppo_grad)"""
    return torch.zeros(_lib.PPO_SCRATCH_BYTES // 8, dtype=torch.float64, device=device)


def _ppo_flags(op, *, value_clipping, reward_scaling, masked_policy, illegal_stat=False, obs_dtype=None) -> int:
    """BrlPpoParams.flags of `op`; obs_dtype = the observations' dtype (None: the op reads none)"""
    try:
        oflag = {None: 0, torch.float32: 0, torch.uint8: _lib.PPO_OBS_U8, torch.bool: _lib.PPO_OBS_U8,
                 torch.bfloat16: _lib.PPO_OBS_BF16}[obs_dtype]
    except KeyError:
        raise _lib.BrlError(f"{op}: observation dtype {obs_dtype} not supported") from None
    return (_lib.PPO_VALUE_CLIPPING if value_clipping else 0) | (_lib.PPO_REWARD_SCALING if reward_scaling else 0) | \
        (0 if masked_policy else _lib.PPO_UNMASKED_POLICY) | (_lib.PPO_ILLEGAL_STAT if illegal_stat else 0) | oflag


def _adam_params(n, step, lr, beta1, beta2, eps, max_grad_norm):
    return _lib.BrlAdamParams(int(n), int(step), float(lr), float(beta1), float(beta2), float(eps), float(max_grad_norm))


def ppo_loss(logits, value, index, mask, action, old_log_prob, old_value, adv, targets, dlogits, dvalue, stats, scratch,
             *, clip_eps, ent_coef, vf_coef, illegal_l2_coef=0.0, value_clipping=True, reward_scaling=False,
             masked_policy=True) -> None:
    """_loss_fn of src/update.py:91-162 + its gradient w.r.t. (logits, value) for one minibatch."""
    flags = _ppo_flags("ppo_loss", value_clipping=value_clipping, reward_scaling=reward_scaling, masked_policy=masked_policy)
    p = _lib.BrlPpoParams(int(logits.shape[0]), int(action.numel()), float(clip_eps), float(ent_coef), float(vf_coef),
                          float(illegal_l2_coef), flags, 0)
    _call("brl_ppo_loss", [_ptr(logits), _ptr(value), _ptr(index), _ptr(mask), _ptr(action), _ptr(old_log_prob),
                           _ptr(old_value), _ptr(adv), _ptr(targets), _ptr(dlogits), _ptr(dvalue), _ptr(stats),
                           _ptr(scratch)], p)


def adam_clip(params, grads, m, v, scratch, *, step: int, lr: float, beta1=0.9, beta2=0.999, eps=1e-5,
              max_grad_norm=0.0, sumsq: Optional[torch.Tensor] = None) -> None:
    """optax.chain(clip_by_global_norm, adam) on flat fp32 buffers, in place (ppo.py:195-211).  `sumsq` (f64[1], e.g.
    `acc[14:15]` after `ppo_grad`): the gradient's sum of squares is already known, skip the pass that forms it."""
    p = _adam_params(params.numel(), step, lr, beta1, beta2, eps, max_grad_norm)
    if sumsq is not None:
        if sumsq.dtype != torch.float64:
            raise _lib.BrlError("adam_clip: sumsq must be float64")
        _call("brl_adam_apply", [_ptr(params), _ptr(grads), _ptr(m), _ptr(v), _ptr(sumsq)], p)
    else:
        _call("brl_adam_clip", [_ptr(params), _ptr(grads), _ptr(m), _ptr(v), _ptr(scratch)], p)


def mlp_num_params() -> int:
    return int(_lib.load().brl_mlp_num_params())


def mlp_pack_train(flat_params: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Flat fp32 parameters (optim.flatten_params order) -> the training blob of `ppo_grad`: W[in, out] as bf16 hi / lo in
    haiku's orientation + fp32 biases.  Once per parameter set; `mlp_adam_step` keeps it current inside the update loop."""
    L = _lib.load()
    if flat_params.dtype != torch.float32 or flat_params.numel() != L.brl_mlp_num_params():
        raise _lib.BrlError("mlp_pack_train needs the flat fp32 parameter buffer of the DeepMind MLP")
    if out is None:
        out = torch.empty(L.brl_mlp_train_blob_bytes(), dtype=torch.uint8, device=flat_params.device)
    _call("brl_mlp_pack_train", [_ptr(flat_params), _ptr(out)], _params(0))
    return out


def mlp_adam_step(params, grads, m, v, sumsq, blob, *, step: int, lr: float, beta1=0.9, beta2=0.999, eps=1e-5,
                  max_grad_norm=0.0) -> None:
    """optax.chain(clip_by_global_norm, adam) on the flat MLP parameters, in place, and the training blob refreshed in
    the same pass (ppo.py:195-211, src/update.py:168-169).  `sumsq`: f64[1] = `acc[14:15]` after `ppo_grad`."""
    if sumsq.dtype != torch.float64:
        raise _lib.BrlError("mlp_adam_step: sumsq must be float64")
    p = _adam_params(params.numel(), step, lr, beta1, beta2, eps, max_grad_norm)
    _call("brl_mlp_adam_step", [_ptr(params), _ptr(grads), _ptr(m), _ptr(v), _ptr(sumsq), _ptr(blob)], p)


def mlp_train_scratch(batch: int, device) -> torch.Tensor:
    return torch.empty(_lib.load().brl_mlp_train_scratch_bytes(batch), dtype=torch.uint8, device=device)


def _anchor_args(op, anchor_logits, kl_coef):
    if (anchor_logits is None) != (kl_coef is None):
        raise _lib.BrlError(f"{op}: anchor_logits and kl_coef go together")


def ppo_grad(obs, blob, scratch, index, mask, action, old_log_prob, old_value, adv, targets, grads, stats, acc, *, clip_eps,
             ent_coef, vf_coef, illegal_l2_coef=0.0, value_clipping=True, reward_scaling=False, masked_policy=True,
             illegal_stat: bool = True, tune: int = 0, anchor_logits: Optional[torch.Tensor] = None,
             kl_coef: Optional[torch.Tensor] = None) -> None:
    """One minibatch of jax.value_and_grad(_loss_fn) (src/update.py:91-167): take(index), forward, loss, backward
    through the MLP on tcgen05 -> flat fp32 gradients (+ the loss statistics of `ppo_loss`).  `illegal_stat=False` (only
    honoured with illegal_l2_coef == 0): skip the logged illegal_action_loss (stats[6] = NaN), ~19 us per call.
    `anchor_logits` (f32 [total, 38], an anchor net's logits for every trajectory row) with `kl_coef` (CUDA f32[1]): add
    kl_coef * mean KL(policy || anchor) to the loss (brl_ppo_grad_anchored); stats[7] = that mean KL."""
    L = _lib.load()
    B = int(index.shape[0]) if index is not None else int(obs.shape[0])
    if obs.dtype == torch.bool:
        obs = obs.view(torch.uint8)
    flags = _ppo_flags("ppo_grad", value_clipping=value_clipping, reward_scaling=reward_scaling, masked_policy=masked_policy,
                       illegal_stat=illegal_stat, obs_dtype=obs.dtype)
    if scratch.numel() < L.brl_mlp_train_scratch_bytes(B) or blob.numel() < L.brl_mlp_train_blob_bytes():
        raise _lib.BrlError("ppo_grad: scratch / blob too small (ops.mlp_train_scratch, ops.mlp_pack_train)")
    _check_flat_grads("ppo_grad", grads)
    _anchor_args("ppo_grad", anchor_logits, kl_coef)
    p = _lib.BrlPpoParams(B, int(action.numel()), float(clip_eps), float(ent_coef), float(vf_coef), float(illegal_l2_coef),
                          flags, int(tune))
    buffers = [_ptr(obs), _ptr(blob), _ptr(scratch), _ptr(index), _ptr(mask), _ptr(action), _ptr(old_log_prob),
               _ptr(old_value), _ptr(adv), _ptr(targets), _ptr(grads), _ptr(stats), _ptr(acc)]
    if anchor_logits is None:
        _call("brl_ppo_grad", buffers, p)
        return
    if anchor_logits.dtype != torch.float32 or anchor_logits.numel() != action.numel() * NUM_ACTIONS:
        raise _lib.BrlError("ppo_grad: anchor_logits must be float32[total, 38] (one row per trajectory row)")
    if kl_coef.dtype != torch.float32 or kl_coef.numel() != 1:
        raise _lib.BrlError("ppo_grad: kl_coef must be a float32[1] device scalar")
    _call("brl_ppo_grad_anchored", buffers + [_ptr(anchor_logits), _ptr(kl_coef)], p)


# ---- population training: K learners' optimizer steps in the launches of one (brl_ppo_grad_grouped) ----------------------
def ppo_grad_grouped_scratch_bytes(n_learners: int, batch: int) -> int:
    return _size_query("brl_ppo_grad_grouped_scratch_bytes", n_learners, batch)


def mlp_param_stride() -> int:
    """floats between two learners' rows of a population's [K, stride] parameter / gradient / moment buffers (a learner
    uses the first mlp_num_params() of its row)"""
    return _size_query("brl_mlp_param_stride")


def ppo_trajectory_row(obs, index, mask, action, old_log_prob, old_value, adv, targets) -> list:
    """One learner's row of the trajectory table of `ppo_grad_grouped`: the device addresses of its `ppo_grad` buffers
    (index may be None = identity).  The tensors must stay alive while a call that reads the table is in flight."""
    if obs.dtype == torch.bool:
        obs = obs.view(torch.uint8)
    return [_ptr(obs), _ptr(index) or 0, _ptr(mask), _ptr(action), _ptr(old_log_prob), _ptr(old_value), _ptr(adv), _ptr(targets)]


def ppo_grad_grouped(traj, coefs, blob, scratch, grads, stats, acc, *, batch: int, obs_dtype, value_clipping=True,
                     reward_scaling=False, masked_policy=True, illegal_stat: bool = True, tune: int = 0,
                     anchor_logits: Optional[torch.Tensor] = None, kl_coef: Optional[torch.Tensor] = None) -> None:
    """`ppo_grad` for K learners in one set of launches.  traj: CUDA int64[K, 8] rows of `ppo_trajectory_row`; coefs: CUDA
    float32[K, 4] = (clip_eps, ent_coef, vf_coef, illegal_l2_coef) per learner; blob: uint8[K, mlp_train_blob_bytes];
    grads: float32[K, mlp_param_stride]; stats: float32[K, 8]; acc: float64[K, PPO_SCRATCH_BYTES / 8], whose row k holds
    learner k's |grads|^2 at element 14 on return.  Every learner's minibatch has `batch` rows and observations of
    `obs_dtype`; learner k's results are bit-identical to `ppo_grad` with its own buffers and coefficients.
    `anchor_logits` (CUDA int64[K]: the device address of learner k's f32 anchor logits [total_k, 38]) with `kl_coef` (CUDA
    float32[K]): each learner's KL term, as `ppo_grad(..., anchor_logits=, kl_coef=)` (brl_ppo_grad_grouped_anchored)."""
    L = _lib.load()
    K = int(traj.shape[0]) if traj.dim() == 2 else -1
    if traj.dtype != torch.int64 or traj.dim() != 2 or traj.shape[1] != 8:
        raise _lib.BrlError("ppo_grad_grouped: traj must be int64[K, 8] (ops.ppo_trajectory_row)")
    if K > _lib.MAX_LEARNERS:
        raise _lib.BrlError(f"ppo_grad_grouped: at most {_lib.MAX_LEARNERS} learners")
    if coefs.dtype != torch.float32 or tuple(coefs.shape) != (K, 4):
        raise _lib.BrlError("ppo_grad_grouped: coefs must be float32[K, 4]")
    n, nb = mlp_param_stride(), L.brl_mlp_train_blob_bytes()
    if grads.dtype != torch.float32 or grads.numel() != K * n or stats.dtype != torch.float32 or stats.numel() != K * 8:
        raise _lib.BrlError("ppo_grad_grouped: grads must be float32[K, mlp_param_stride], stats float32[K, 8]")
    if blob.numel() != K * nb or scratch.numel() < ppo_grad_grouped_scratch_bytes(K, batch) or \
            acc.dtype != torch.float64 or acc.numel() != K * (_lib.PPO_SCRATCH_BYTES // 8):
        raise _lib.BrlError("ppo_grad_grouped: blob must be uint8[K, mlp_train_blob_bytes], acc float64[K, PPO_SCRATCH_BYTES / 8], "
                            "scratch ppo_grad_grouped_scratch_bytes(K, batch)")
    flags = _ppo_flags("ppo_grad_grouped", value_clipping=value_clipping, reward_scaling=reward_scaling, masked_policy=masked_policy,
                       illegal_stat=illegal_stat, obs_dtype=obs_dtype)
    _anchor_args("ppo_grad_grouped", anchor_logits, kl_coef)
    p = _lib.BrlPpoGroupedParams(int(batch), K, flags, int(tune), 0)
    buffers = [_ptr(traj), _ptr(coefs), _ptr(blob), _ptr(scratch), _ptr(grads), _ptr(stats), _ptr(acc)]
    if anchor_logits is None:
        _call("brl_ppo_grad_grouped", buffers, p)
        return
    if anchor_logits.dtype != torch.int64 or anchor_logits.numel() != K or kl_coef.dtype != torch.float32 or kl_coef.numel() != K:
        raise _lib.BrlError("ppo_grad_grouped: anchor_logits must be int64[K] device addresses, kl_coef float32[K]")
    _call("brl_ppo_grad_grouped_anchored", buffers + [_ptr(anchor_logits), _ptr(kl_coef)], p)


def mlp_adam_step_grouped(params, grads, m, v, acc, blob, *, steps, lrs, max_grad_norms, beta1=0.9, beta2=0.999,
                          eps=1e-5) -> None:
    """`mlp_adam_step` for K learners in one launch: params / grads / m / v float32[K, mlp_param_stride], blob
    uint8[K, mlp_train_blob_bytes], acc = `ppo_grad_grouped`'s float64[K, PPO_SCRATCH_BYTES / 8].  steps, lrs,
    max_grad_norms (and beta1, beta2, eps when given as sequences): one entry per learner."""
    L = _lib.load()
    K = len(steps)
    if len(lrs) != K or len(max_grad_norms) != K:
        raise _lib.BrlError("mlp_adam_step_grouped: steps, lrs and max_grad_norms need one entry per learner")
    if K > _lib.MAX_LEARNERS:
        raise _lib.BrlError(f"mlp_adam_step_grouped: at most {_lib.MAX_LEARNERS} learners")
    n, stride = L.brl_mlp_num_params(), mlp_param_stride()
    for name, t in (("params", params), ("grads", grads), ("m", m), ("v", v)):
        if t.dtype != torch.float32 or t.numel() != K * stride:
            raise _lib.BrlError(f"mlp_adam_step_grouped: {name} must be float32[K, mlp_param_stride]")
    if acc.dtype != torch.float64 or acc.numel() != K * (_lib.PPO_SCRATCH_BYTES // 8) or \
            blob.numel() != K * L.brl_mlp_train_blob_bytes():
        raise _lib.BrlError("mlp_adam_step_grouped: acc must be float64[K, PPO_SCRATCH_BYTES / 8], blob uint8[K, mlp_train_blob_bytes]")

    def per(x):
        return list(x) if isinstance(x, (list, tuple)) else [x] * K
    b1, b2, ep = per(beta1), per(beta2), per(eps)
    p = (_lib.BrlAdamParams * K)(*[_adam_params(n, steps[k], lrs[k], b1[k], b2[k], ep[k], max_grad_norms[k]) for k in range(K)])
    _call("brl_mlp_adam_step_grouped", [_ptr(params), _ptr(grads), _ptr(m), _ptr(v), _ptr(acc), _ptr(blob)], p)


def sl_examples(table, calls, offsets, traj, obs, mask, label, *, position=None, position_out=None, seed=0, step=0,
                env_offset=0) -> None:
    """make_dataset of sl.py:100-117 for a batch: example b replays trajectory traj[b] up to its call `position[b]` (drawn
    uniformly in-kernel from Philox(seed; env_offset + b, step) when `position` is None) and gets the observation and
    legal mask of the player to act, and that call as its label.  `obs` dtype: float32, uint8 / bool or bfloat16."""
    if offsets.dtype != torch.int64 or calls.dtype != torch.uint8 or traj.dtype != torch.int32:
        raise _lib.BrlError("sl_examples: calls must be uint8, offsets int64, traj int32")
    n_traj = int(offsets.shape[0]) - 1
    flags = obs_flag(obs.dtype)
    _call("brl_sl_examples", [_ptr(table), _ptr(calls), _ptr(offsets), _ptr(traj), _ptr(position), _ptr(obs), _ptr(mask),
                              _ptr(label), _ptr(position_out), None],
          _params(traj.shape[0], flags=flags, seed=seed, step=step, env_offset=env_offset, n_deals=n_traj))


def sl_check(table, calls, offsets, status: torch.Tensor) -> None:
    """Replay every whole auction once: status[t] = _lib.SL_OK / SL_ILLEGAL / SL_EARLY_END / SL_NOT_ENDED."""
    n_traj = int(offsets.shape[0]) - 1
    _call("brl_sl_examples", [_ptr(table), _ptr(calls), _ptr(offsets), None, None, None, None, None, None, _ptr(status)],
          _params(n_traj, flags=_lib.F_SL_CHECK, n_deals=n_traj))


def sl_acc(device) -> torch.Tensor:
    """f64[16] accumulators of sl_grad / sl_eval (element 14 = sum of squares of the gradient after sl_grad)"""
    return torch.zeros(_lib.SL_ACC_BYTES // 8, dtype=torch.float64, device=device)


def _head_params(name, B, obs, scratch, blob, ent_coef, tiles=0):
    """obs as the loss-head ops on BrlSlParams read it (bool as uint8), and their params; after the op's own input checks"""
    L = _lib.load()
    if obs.dtype == torch.bool:
        obs = obs.view(torch.uint8)
    if scratch.numel() < L.brl_mlp_train_scratch_bytes(B) or blob.numel() < L.brl_mlp_train_blob_bytes():
        raise _lib.BrlError(f"{name}: scratch / blob too small (ops.mlp_train_scratch, ops.mlp_pack_train)")
    if tiles & ~(CV_WIDE_FORWARD | CV_NARROW_BACKWARD):
        raise _lib.BrlError(f"{name}: tiles takes CV_WIDE_FORWARD / CV_NARROW_BACKWARD only")
    return obs, _lib.BrlSlParams(B, float(ent_coef), obs_flag(obs.dtype) | tiles)


def _check_flat_grads(name, grads):
    if grads.dtype != torch.float32 or grads.numel() != _lib.load().brl_mlp_num_params():
        raise _lib.BrlError(f"{name}: grads must be the flat fp32 gradient buffer")


def _check_sl_inputs(name, mask, label):
    if label.dtype != torch.int32 or mask.dtype != torch.uint8:
        raise _lib.BrlError(f"{name}: label must be int32 and mask uint8")


def sl_grad(obs, blob, scratch, mask, label, grads, stats, acc, *, ent_coef=0.0) -> None:
    """One minibatch of value_and_grad(loss) of sl.py:169-184 through the MLP on tcgen05 -> flat fp32 gradients and
    stats[:5] = {total_loss, target_loss, entropy, accuracy, illegal_actions_prob} of the parameters before the step."""
    _check_sl_inputs("sl_grad", mask, label)
    obs, p = _head_params("sl_grad", int(label.shape[0]), obs, scratch, blob, ent_coef)
    _check_flat_grads("sl_grad", grads)
    _call("brl_sl_grad", [_ptr(obs), _ptr(blob), _ptr(scratch), _ptr(mask), _ptr(label), _ptr(grads), _ptr(stats), _ptr(acc)], p)


def sl_eval(obs, blob, scratch, mask, label, stats, acc, *, ent_coef=0.0) -> None:
    """sl_grad's statistics without the backward (accuracy, sl.py:186-194; test metrics, sl.py:288-301)."""
    _check_sl_inputs("sl_eval", mask, label)
    obs, p = _head_params("sl_eval", int(label.shape[0]), obs, scratch, blob, ent_coef)
    _call("brl_sl_eval", [_ptr(obs), _ptr(blob), _ptr(scratch), _ptr(mask), _ptr(label), _ptr(stats), _ptr(acc)], p)


CV_WIDE_FORWARD, CV_NARROW_BACKWARD = 1 << 16, 1 << 17  # brl_cv_grad's tile-width experiment bits (BRL_CV_*)


def _check_cv_inputs(name, obs, gain):
    B = int(gain.shape[0])
    if gain.dtype != torch.float32 or tuple(gain.shape) != (B, NUM_ACTIONS):
        raise _lib.BrlError(f"{name}: gain must be float32 [B, 38] (NaN for an illegal call)")
    if tuple(obs.shape) != (B, OBS_DIM):
        raise _lib.BrlError(f"{name}: obs must be [B, 480] with B = gain.shape[0]")


def cv_grad(obs, blob, scratch, gain, grads, stats, acc, *, ent_coef=0.0, tiles=0) -> None:
    """One minibatch of the call-value policy-improvement loss (DESIGN.md f17) through the MLP on tcgen05: gain f32[B, 38]
    (IMPs, NaN = illegal), loss = -mean(sum_a pi_a g_a) / 24 - ent_coef * mean entropy -> flat fp32 gradients, stats[8]
    (include/brl_b200.h brl_cv_grad) and acc[14] = sum of squares of the gradient (sl_acc's buffer).  `tiles`: the
    CV_WIDE_FORWARD / CV_NARROW_BACKWARD experiment bits (0: the measured tile widths)."""
    _check_cv_inputs("cv_grad", obs, gain)
    obs, p = _head_params("cv_grad", int(gain.shape[0]), obs, scratch, blob, ent_coef, tiles)
    _check_flat_grads("cv_grad", grads)
    _call("brl_cv_grad", [_ptr(obs), _ptr(blob), _ptr(scratch), _ptr(gain), _ptr(grads), _ptr(stats), _ptr(acc)], p)


def cv_eval(obs, blob, scratch, gain, stats, acc, *, ent_coef=0.0, tiles=0) -> None:
    """cv_grad's statistics without the backward (bit-equal to cv_grad's on the same inputs)."""
    _check_cv_inputs("cv_eval", obs, gain)
    obs, p = _head_params("cv_eval", int(gain.shape[0]), obs, scratch, blob, ent_coef, tiles)
    _call("brl_cv_eval", [_ptr(obs), _ptr(blob), _ptr(scratch), _ptr(gain), _ptr(stats), _ptr(acc)], p)


def gather_rows(src: torch.Tensor, index: torch.Tensor, dst: torch.Tensor) -> None:
    """dst[b] = src[index[b]] over the leading axis (minibatch take, src/update.py:194-199)."""
    row_bytes = src[0].numel() * src.element_size()
    _call("brl_gather_rows", [_ptr(src), _ptr(index), _ptr(dst)], _params(index.shape[0], k_steps=row_bytes))


def eval_act_log(logits_team1, logits_team2, mask, current_player, terminated, action, acc, indicator_bids=False) -> None:
    """masked argmax of the acting team's logits + update_log_info (src/evaluation.py:236-385, 650-745)."""
    n = logits_team1.shape[0]
    _call("brl_eval_act_log", [_ptr(logits_team1), _ptr(logits_team2), _ptr(mask), _ptr(current_player), _ptr(terminated),
                               _ptr(action), _ptr(acc)],
          _params(n, flags=_lib.F_EVAL_INDICATOR_BIDS if indicator_bids else 0))


def eval_summary(acc, cum_return, step_count, table_a, table_b, sums) -> None:
    """table_* = (last_bid i32, last_bidder i32, call_x u8, call_xx u8, rewards f32[n,4] | None, pass_num i32 | None);
    table_b may be None (single-table evaluate).  sums f64[brl_eval_num_sums()] += partial sums."""
    tb = table_b if table_b is not None else (None,) * 6
    _call("brl_eval_summary", [_ptr(acc), _ptr(cum_return), _ptr(step_count)] + [_ptr(t) for t in table_a] +
          [_ptr(t) for t in tb] + [_ptr(sums)], _params(cum_return.shape[0]))


_FIELD_SPECS = (("deal", torch.int32, ()), ("dealer", torch.int32, ()), ("shuffled_players", torch.int8, (4,)),
                ("vul", torch.uint8, (2,)), ("last_bid", torch.int32, ()), ("last_bidder", torch.int32, ()),
                ("call_x", torch.uint8, ()), ("call_xx", torch.uint8, ()), ("pass_num", torch.int32, ()),
                ("step_count", torch.int32, ()), ("rng_key", torch.int64, ()))


def state_fields(state: torch.Tensor) -> dict:
    """Unpack the private pgx-style fields brl reads (src/evaluation.py:97-112, 465-495)."""
    n = state.shape[1]
    out = {name: torch.empty((n,) + shape, dtype=dt, device=state.device) for name, dt, shape in _FIELD_SPECS}
    _call("brl_state_fields", [_ptr(state)] + [_ptr(out[name]) for name, _, _ in _FIELD_SPECS],
              _params(n, stride=state.shape[1]))
    return out


# ---- self-play league over a pool of nets (workspace/eval_selfplay_league.py) ----------------------------------------
def _size_query(name: str, *args) -> int:
    fn = getattr(_lib.load(), name)
    fn.restype, fn.argtypes = _lib.C.c_int64, [_lib.C.c_int64] * len(args)
    return int(fn(*args))


def mlp_pool_stride() -> int:
    """bytes between two nets of a pool blob (a packed blob, padded to keep every section's TMA alignment)"""
    return _size_query("brl_mlp_pool_stride")


def model_rows_capacity(n_envs: int, n_models: int) -> int:
    """rows `model_rows` may need for n_envs envs over n_models nets (each group padded to 256 rows)"""
    return _size_query("brl_model_rows_capacity", n_envs, n_models)


def policy_grouped_scratch_bytes(n_envs: int, n_models: int) -> int:
    return _size_query("brl_policy_grouped_scratch_bytes", n_envs, n_models)


def mlp_pack_pool(params_list, pack_one) -> torch.Tensor:
    """Stack the packed blobs of `params_list` as u8[M, mlp_pool_stride()]; `pack_one(params, out)` packs one net into
    `out` (ForwardPass.pack_into, i.e. mlp_pack(out=...))."""
    if not params_list:
        raise _lib.BrlError("mlp_pack_pool: empty pool")
    dev = next(iter(params_list[0].values()))["w"].device
    pool = torch.zeros((len(params_list), mlp_pool_stride()), dtype=torch.uint8, device=dev)
    size = _lib.load().brl_mlp_packed_bytes()
    for m, params in enumerate(params_list):
        pack_one(params, pool[m, :size])
    return pool


def _check_pool(who: str, pool: torch.Tensor, n_nets: Optional[int] = None, min_nets: int = 0, suffix: str = "") -> None:
    """pool u8[M, mlp_pool_stride()], with M = n_nets when given and M >= min_nets"""
    if pool.dim() != 2 or pool.dtype != torch.uint8 or pool.shape[1] != mlp_pool_stride() or pool.shape[0] < min_nets or \
            (n_nets is not None and pool.shape[0] != n_nets):
        raise _lib.BrlError(f"{who}: pool must be u8[{'M' if n_nets is None else n_nets}, mlp_pool_stride()] (ops.mlp_pack_pool)"
                            + suffix)


def _check_env_models(who: str, env_models: torch.Tensor, n: int) -> None:
    if env_models.dtype != torch.int32 or tuple(env_models.shape) not in ((n, 2), (n, 4)):
        raise _lib.BrlError(f"{who}: env_models must be int32 [n, 2] (by team) or [n, 4] (by player)")


def _check_deal_table(who: str, table: torch.Tensor) -> None:
    if table.dtype != torch.uint8 or table.dim() != 2 or table.shape[1] != 48:
        raise _lib.BrlError(f"{who}: the deal table must be u8 [n_deals, 48]")


def model_rows(current_player: torch.Tensor, done: Optional[torch.Tensor], env_models: torch.Tensor, rows: torch.Tensor,
               counts: torch.Tensor, offsets: torch.Tensor, block_model: torch.Tensor) -> None:
    """Live envs (done == 0) grouped by the net that acts there: env_models[i, 0] for players 0/1, [i, 1] for players 2/3,
    or, with env_models int32[n, 4], env_models[i, player] for each player id (BRL_F_PLAYER_MODELS).  Net m's rows are rows[offsets[m] : offsets[m] + counts[m]], padded with -1 to offsets[m + 1]; offsets[M] is the padded
    row count and block_model the net of each 256-row block.  A live env whose id is outside [0, M) makes offsets[M] = -1:
    the grouping is invalid, and the caller's read of offsets[M] (which sizes the forward) must raise."""
    n_models = counts.shape[0]
    _check_env_models("model_rows", env_models, current_player.shape[0])
    if offsets.shape[0] != n_models + 1 or rows.shape[0] < model_rows_capacity(current_player.shape[0], n_models):
        raise _lib.BrlError("model_rows: offsets must hold M + 1 entries and rows model_rows_capacity(n, M)")
    flags = _lib.F_PLAYER_MODELS if env_models.shape[1] == 4 else 0
    _call("brl_model_rows", [_ptr(current_player), _ptr(done), _ptr(env_models), _ptr(rows), _ptr(counts), _ptr(offsets),
                             _ptr(block_model)], _params(current_player.shape[0], k_steps=n_models, flags=flags))


def policy_act_grouped(obs_bf16: torch.Tensor, pool: torch.Tensor, scratch: torch.Tensor, mask: Optional[torch.Tensor],
                       action: torch.Tensor, rows: torch.Tensor, block_model: torch.Tensor,
                       logits: Optional[torch.Tensor] = None, *, n_rows: Optional[torch.Tensor] = None,
                       single_bf16: bool = False, tune: int = 0) -> None:
    """`policy_act_rows` (masked argmax) for the padded, net-grouped `rows` of `model_rows`, net block_model[b] on rows
    [256 b, 256 b + 256), all nets of `pool` (u8[M, mlp_pool_stride()]) in one forward.  n_rows[0] is the padded row count
    (`offsets[M:]` of `model_rows`), read on the device only: rows from n_rows[0] on are not read, and the call is sized
    (and its launch path chosen) for rows.shape[0].  Without n_rows the rows end at the count (rows = rows[:offsets[M]]).
    rows / block_model / n_rows must come from `model_rows` with the same M (device data, not checked here)."""
    n = rows.shape[0]
    if n == 0:
        return
    if obs_bf16.dtype != torch.bfloat16 or rows.dtype != torch.int32 or block_model.dtype != torch.int32:
        raise _lib.BrlError("policy_act_grouped needs a bf16 observation and int32 rows / block_model")
    if n_rows is None:
        n_rows = torch.full((1,), n, dtype=torch.int32, device=rows.device)
    if not n_rows.is_cuda or n_rows.dtype != torch.int32 or n_rows.numel() < 1:
        raise _lib.BrlError("policy_act_grouped: n_rows must be a CUDA int32 tensor holding the padded row count (offsets[M:])")
    _check_pool("policy_act_grouped", pool)
    if scratch.numel() < _lib.load().brl_mlp_rows_scratch_bytes(n):
        raise _lib.BrlError("policy_act_grouped: scratch too small (ops.policy_grouped_scratch_bytes)")
    _call("brl_policy_act_grouped", [_ptr(obs_bf16), _ptr(pool), _ptr(scratch), _ptr(mask), _ptr(action), _ptr(rows),
                                     _ptr(block_model), _ptr(logits), _ptr(n_rows)],
          _params(n, k_steps=pool.shape[0], flags=(F_MLP_BF16 if single_bf16 else 0) | tune))


def match_stats_ranges(x: torch.Tensor, offsets: torch.Tensor, sums: torch.Tensor) -> None:
    """sums[p, :4] += match_stats of x[offsets[p]:offsets[p + 1]] for every range p (offsets int64[P + 1], sums f64[P, 8])."""
    if offsets.dtype != torch.int64 or sums.dtype != torch.float64 or tuple(sums.shape) != (offsets.shape[0] - 1, 8):
        raise _lib.BrlError("match_stats_ranges: offsets must be int64[P + 1] and sums float64[P, 8]")
    _call("brl_match_stats_ranges", [_ptr(x), _ptr(offsets), _ptr(sums)], _params(sums.shape[0]))


# ---- a whole duplicate match as one call (eval.py:53, src/evaluation.py:69-204) -------------------------------------------
def duplicate_match_scratch_bytes(n_envs: int, n_models: int) -> int:
    return _size_query("brl_duplicate_match_scratch_bytes", n_envs, n_models)


def duplicate_match_graph_builds() -> int:
    """graphs brl_duplicate_match has captured and instantiated in this process (a repeated call with the same buffers and
    parameters relaunches its cached graph)"""
    fn = _lib.load().brl_duplicate_match_graph_builds
    fn.restype, fn.argtypes = _lib.C.c_longlong, []
    return int(fn())


def duplicate_match(keys: torch.Tensor, table: torch.Tensor, pool: torch.Tensor, scratch: torch.Tensor, cum_return: torch.Tensor,
                    sums: torch.Tensor, status: torch.Tensor, *, env_models: Optional[torch.Tensor] = None,
                    range_offsets: Optional[torch.Tensor] = None, table_a: Optional[TableInfoBuffers] = None,
                    table_b: Optional[TableInfoBuffers] = None, single_bf16: bool = False, tune: int = 0,
                    illegal_penalty: float = -1.0, illegal_bonus: float = 1.0,
                    system_hist: Optional[torch.Tensor] = None) -> None:
    """Play duplicate_evaluate's whole loop (src/evaluation.py:93-201) for every env of `keys` in one call, with the loop on
    the device: env e plays net env_models[e, 0] of `pool` on players 0/1 against env_models[e, 1] on 2/3 (default: net 0
    against net 1, M must be 2), or with env_models int32[n, 4] net env_models[e, p] on player p (BRL_F_PLAYER_MODELS: each
    partner may be a different net).  Writes cum_return f32[n], adds the match sums to `sums` (f64[P, 8] over the ranges of
    `range_offsets` int64[P + 1], or f64[8] for the whole batch), the status (int32[1], _lib.MATCH_*) and, when given, the
    final Table_info of both tables.  `system_hist` (u32 [M, 75, 38, 96], see `system_stats`): every decision of the match is
    added to the histogram of the net that made it.  Nothing is read back to the host; read `status` with the sums."""
    n, M = int(keys.shape[0]), int(pool.shape[0]) if pool.dim() == 2 else 0
    if env_models is None and M != 2:
        raise _lib.BrlError(f"duplicate_match: without env_models the pool must hold 2 nets, got {M}")
    if env_models is not None:
        _check_env_models("duplicate_match", env_models, n)
    player_models = env_models is not None and env_models.shape[1] == 4
    P = 0
    if range_offsets is not None:
        P = int(range_offsets.shape[0]) - 1
        if range_offsets.dtype != torch.int64 or P < 1 or tuple(sums.shape) != (P, 8):
            raise _lib.BrlError("duplicate_match: range_offsets must be int64[P + 1] with sums float64[P, 8]")
    elif sums.numel() != 8:
        raise _lib.BrlError("duplicate_match: without range_offsets sums is float64[8]")
    if sums.dtype != torch.float64 or cum_return.dtype != torch.float32 or status.dtype != torch.int32:
        raise _lib.BrlError("duplicate_match: sums must be float64, cum_return float32 and status int32")
    _check_pool("duplicate_match", pool)
    if scratch.numel() < duplicate_match_scratch_bytes(n, M):
        raise _lib.BrlError("duplicate_match: scratch too small (ops.duplicate_match_scratch_bytes)")
    if (table_a is None) != (table_b is None):
        raise _lib.BrlError("duplicate_match: give both Table_info outputs or neither")
    if system_hist is not None:
        _check_system_hist("duplicate_match", system_hist, M)
    infos = table_a.ptrs() + table_b.ptrs() if table_a is not None else [None] * 12
    _call("brl_duplicate_match", [_ptr(keys), _ptr(table), _ptr(pool), _ptr(env_models), _ptr(range_offsets), _ptr(scratch),
                                  _ptr(cum_return), _ptr(sums), _ptr(status)] + infos + [_ptr(system_hist)],
          _params(n, k_steps=M, step=P, n_deals=table.shape[0],
                  flags=(F_MLP_BF16 if single_bf16 else 0) | (_lib.F_PLAYER_MODELS if player_models else 0) | tune,
                  illegal_penalty=illegal_penalty, illegal_bonus=illegal_bonus))


# ---- a whole evaluation as one call (ppo.py:365-374; src/evaluation.py:11-66, 207-1032) -----------------------------------
def evaluate_match_scratch_bytes(n_envs: int, mode: int, partner: bool = False) -> int:
    """scratch bytes of `evaluate_match` for n_envs envs in `mode`, with or without the partner's net in the pool"""
    name = "brl_evaluate_match_partner_scratch_bytes" if partner else "brl_evaluate_match_scratch_bytes"
    return _size_query(name, n_envs, mode)


def evaluate_match(keys: torch.Tensor, table: torch.Tensor, pool: torch.Tensor, scratch: torch.Tensor, cum_return: torch.Tensor,
                   status: torch.Tensor, *, mode: int, acc: Optional[torch.Tensor] = None, sums: Optional[torch.Tensor] = None,
                   table_a: Optional[TableInfoBuffers] = None, table_b: Optional[TableInfoBuffers] = None,
                   final_state: Optional[torch.Tensor] = None, final: Optional[EnvOutputs] = None, free_run: bool = False,
                   partner: bool = False, single_bf16: bool = False, tune: int = 0, illegal_penalty: float = -1.0,
                   illegal_bonus: float = 1.0) -> None:
    """Play a whole evaluation (make_evaluate's duplicate_evaluate / evaluate, or make_simple_evaluate) for every env of `keys`
    in one call, with the loop on the device.  `pool` u8[2, mlp_pool_stride()]: net 0 is team 1 / the actor, net 1 team 2 / the
    opponent (not read with free_run).  `mode` = _lib.EVAL_MATCH_*:
      DUPLICATE / SINGLE: writes cum_return f32[n] and acc f32[n, EVAL_ACC_COLS], adds brl_eval_summary's partial sums to `sums`
        (f64[brl_eval_num_sums()]); DUPLICATE writes the final Table_infos when given, SINGLE the final state (`final_state`
        int32[5, n, 4], `final` with a bf16 observation; its rewards = the summed step rewards) when given;
      SIMPLE: cum_return = R, the per-env return of the player to act at the start.
    `partner` (BRL_F_EVAL_PARTNER): `pool` is u8[3, mlp_pool_stride()] and net 2 plays the actor's partner -- player 1 in
    DUPLICATE / SINGLE, the initial player's partner in SIMPLE -- with the scratch of evaluate_match_scratch_bytes(n, mode,
    partner=True).
    `status` (int32[1], _lib.MATCH_*) is written too; nothing is read back to the host."""
    n = int(keys.shape[0])
    if mode not in (_lib.EVAL_MATCH_DUPLICATE, _lib.EVAL_MATCH_SINGLE, _lib.EVAL_MATCH_SIMPLE):
        raise _lib.BrlError(f"evaluate_match: unknown mode {mode}")
    full = mode != _lib.EVAL_MATCH_SIMPLE
    if free_run and not full:
        raise _lib.BrlError("evaluate_match: free_run is a mode of the full-statistics evaluation")
    _check_pool("evaluate_match", pool, 3 if partner else 2, suffix=" with the partner's net" if partner else "")
    if cum_return.dtype != torch.float32 or status.dtype != torch.int32:
        raise _lib.BrlError("evaluate_match: cum_return must be float32 and status int32")
    if full:
        if acc is None or sums is None or acc.dtype != torch.float32 or tuple(acc.shape) != (n, _lib.EVAL_ACC_COLS) or \
                sums.dtype != torch.float64 or sums.numel() != _lib.load().brl_eval_num_sums():
            raise _lib.BrlError("evaluate_match: full statistics need acc float32[n, 76] and sums float64[239]")
    if scratch.numel() < evaluate_match_scratch_bytes(n, mode, partner):
        raise _lib.BrlError("evaluate_match: scratch too small (ops.evaluate_match_scratch_bytes)")
    if (table_a is None) != (table_b is None):
        raise _lib.BrlError("evaluate_match: give both Table_info outputs or neither")
    if (final_state is None) != (final is None):
        raise _lib.BrlError("evaluate_match: give the final state and its outputs together or neither")
    if final is not None and final.observation.dtype != torch.bfloat16:
        raise _lib.BrlError("evaluate_match: the final observation is bf16")
    infos = table_a.ptrs() + table_b.ptrs() if table_a is not None else [None] * 12
    finals = [_ptr(final_state)] + final.ptrs() if final is not None else [None] * 6
    flags = _lib.f_eval_match(mode) | (_lib.F_EVAL_FREE_RUN if free_run else 0) | (F_MLP_BF16 if single_bf16 else 0) | tune
    if partner:
        flags |= _lib.F_EVAL_PARTNER
    _call("brl_evaluate_match", [_ptr(keys), _ptr(table), _ptr(pool), _ptr(scratch), _ptr(cum_return), _ptr(acc), _ptr(sums),
                                 _ptr(status)] + infos + finals,
          _params(n, n_deals=table.shape[0], flags=flags, k_steps=3 if partner else 0, illegal_penalty=illegal_penalty,
                  illegal_bonus=illegal_bonus))


# ---- bidding-system statistics (DESIGN.md f15) ---------------------------------------------------------------------------
SYSTEM_SHAPE = (_lib.SYS_CONTEXTS, NUM_ACTIONS, _lib.SYS_COLS)  # one net's histogram: [context, call, column]


def new_system_hist(n_models: int, device) -> torch.Tensor:
    """A zeroed bidding-system histogram u32 [M, 75, 38, 96] for `system_stats` / `duplicate_match(system_hist=)`."""
    return torch.zeros((n_models,) + SYSTEM_SHAPE, dtype=torch.uint32, device=device)


def system_hist_counts(hist: torch.Tensor) -> torch.Tensor:
    """The u32 cells of a device histogram as int64 (for accumulating calls beyond 2^32 - 1)."""
    return hist.view(torch.int32).to(torch.int64) & 0xFFFFFFFF


def _check_system_hist(who: str, hist: torch.Tensor, n_models: int) -> None:
    if hist.dtype not in (torch.uint32, torch.int32) or tuple(hist.shape) != (n_models,) + SYSTEM_SHAPE:
        raise _lib.BrlError(f"{who}: the system histogram must be u32 [{n_models}, 75, 38, 96] (ops.new_system_hist)")


def system_stats(state: torch.Tensor, table: torch.Tensor, action: torch.Tensor, hist: torch.Tensor, *,
                 done: Optional[torch.Tensor] = None, env_models: Optional[torch.Tensor] = None) -> None:
    """hist += one decision per live env (done == 0; no `done`: every env): the call action[i] of the player to act in
    `state` (before the step), with that player's hand, in the context the earlier calls give it, counted for the net acting
    there -- env_models int32 [n, 2] by team or [n, 4] by player id, as `model_rows` reads them (None: net 0).  `hist` is
    u32 [M, 75, 38, 96]; a call outside 0..37 or a net id outside [0, M) is not counted."""
    n = int(action.shape[0])
    M = int(hist.shape[0]) if hist.dim() == 4 else 0
    _check_system_hist("system_stats", hist, max(M, 1))
    if state.dtype != torch.int32 or state.dim() != 3 or state.shape[0] != STATE_PLANES or state.shape[1] < n:
        raise _lib.BrlError("system_stats: state must be a packed state int32 [5, >= n, 4] (ops.new_state)")
    if action.dtype != torch.int32 or action.dim() != 1:
        raise _lib.BrlError("system_stats: action must be int32 [n]")
    if done is not None and (done.dtype not in (torch.uint8, torch.bool) or tuple(done.shape) != (n,)):
        raise _lib.BrlError("system_stats: done must be uint8 / bool [n]")
    if env_models is not None:
        _check_env_models("system_stats", env_models, n)
    _check_deal_table("system_stats", table)
    flags = _lib.F_PLAYER_MODELS if env_models is not None and env_models.shape[1] == 4 else 0
    _call("brl_system_stats", [_ptr(state), _ptr(table), _ptr(action), _ptr(done), _ptr(env_models), _ptr(hist)],
          _params(n, stride=state.shape[1], k_steps=M, n_deals=table.shape[0], flags=flags))


def system_stats_auctions(table: torch.Tensor, calls: torch.Tensor, offsets: torch.Tensor, hist: torch.Tensor, *,
                          board: Optional[torch.Tensor] = None, dealer: Optional[torch.Tensor] = None) -> None:
    """hist (u32 [1, 75, 38, 96]) += every call of the stored auctions: auction t is calls[offsets[t]:offsets[t + 1]] (u8,
    0..37, the encoding of `sl_examples`) on deal row board[t] (int32; None: row t) with dealer dealer[t] (int8; None: North).
    The calls, the rows and the dealers are checked on the host (one device-to-host copy of each) before any device work."""
    n = int(offsets.shape[0]) - 1
    _check_system_hist("system_stats_auctions", hist, 1)
    if offsets.dtype != torch.int64 or offsets.dim() != 1 or n < 0:
        raise _lib.BrlError("system_stats_auctions: offsets must be int64 [n + 1]")
    if calls.dtype != torch.uint8 or calls.dim() != 1:
        raise _lib.BrlError("system_stats_auctions: calls must be u8 [total]")
    _check_deal_table("system_stats_auctions", table)
    if board is not None and (board.dtype != torch.int32 or tuple(board.shape) != (n,)):
        raise _lib.BrlError("system_stats_auctions: board must be int32 [n]")
    if dealer is not None and (dealer.dtype != torch.int8 or tuple(dealer.shape) != (n,)):
        raise _lib.BrlError("system_stats_auctions: dealer must be int8 [n]")
    if n == 0:
        return
    off = offsets.cpu()
    if int(off[0]) != 0 or bool((off[1:] < off[:-1]).any()) or int(off[-1]) != calls.shape[0]:
        raise _lib.BrlError("system_stats_auctions: offsets must rise from 0 to len(calls)")
    if int(off[-1]) >= 1 << 32:
        raise _lib.BrlError("system_stats_auctions: at most 2^32 - 1 calls per call (a u32 cell could wrap)")
    if calls.numel() and int(calls.max()) >= NUM_ACTIONS:
        raise _lib.BrlError("system_stats_auctions: a call is outside 0..37")
    if board is None and n > table.shape[0]:
        raise _lib.BrlError("system_stats_auctions: without board auction t needs deal row t: the table is too short")
    if board is not None and (int(board.min()) < 0 or int(board.max()) >= table.shape[0]):
        raise _lib.BrlError("system_stats_auctions: a board row is outside the deal table")
    if dealer is not None and (int(dealer.min()) < 0 or int(dealer.max()) > 3):
        raise _lib.BrlError("system_stats_auctions: a dealer is outside 0..3")
    _call("brl_system_stats_auctions", [_ptr(table), _ptr(calls), _ptr(offsets), _ptr(board), _ptr(dealer), _ptr(hist)],
          _params(n, n_deals=table.shape[0]))


# ---- counterfactual call values (DESIGN.md f16) ----------------------------------------------------------------------------
CALL_GAIN_SHAPE = (_lib.SYS_CONTEXTS, NUM_ACTIONS, NUM_ACTIONS, 4)  # one net's gain sums: [context, played, alternative, stat]
CALL_REGRET_SHAPE = (_lib.SYS_CONTEXTS, 4)                          # one net's regret sums: [context, stat]
CALL_RECORD_FIELDS = ("env", "table", "player", "net", "context", "played")


def call_values_scratch_bytes(n_envs: int, n_models: int) -> int:
    return _size_query("brl_call_values_scratch_bytes", n_envs, n_models)


class CallValueRecords:
    """Record buffers of `call_values` for `capacity` decisions: int32 env, table, player, net, context, played [cap], f32
    r[cap, 38] (NaN for an illegal call) and the int64 decision count[1] (also counted beyond the capacity).  With `train`
    also the training examples of DESIGN.md f17: bf16 obs[cap, 480] (the observation the acting net read) and f32
    gain[cap, 38] (g_d(a) in IMPs, NaN where the call is illegal), row k belonging to record k."""

    def __init__(self, capacity: int, device, train: bool = False):
        self.capacity = int(capacity)
        self.count = torch.zeros(1, dtype=torch.int64, device=device)
        for f in CALL_RECORD_FIELDS:
            setattr(self, f, torch.empty(self.capacity, dtype=torch.int32, device=device))
        self.r = torch.empty((self.capacity, NUM_ACTIONS), dtype=torch.float32, device=device)
        self.train = bool(train)
        self.obs = torch.empty((self.capacity, OBS_DIM), dtype=torch.bfloat16, device=device) if train else None
        self.gain = torch.empty((self.capacity, NUM_ACTIONS), dtype=torch.float32, device=device) if train else None

    def ptrs(self):
        return ([_ptr(self.count)] + [_ptr(getattr(self, f)) for f in CALL_RECORD_FIELDS] + [_ptr(self.r)]
                + [_ptr(self.obs), _ptr(self.gain)])


def call_values(keys: torch.Tensor, table: torch.Tensor, pool: torch.Tensor, env_models: torch.Tensor, rewards_a: torch.Tensor,
                rewards_b: torch.Tensor, scratch: torch.Tensor, gain_sums: torch.Tensor, regret_sums: torch.Tensor,
                mismatch: torch.Tensor, status: torch.Tensor, *, records: Optional[CallValueRecords] = None,
                env_offset: int = 0, single_bf16: bool = False, tune: int = 0, illegal_penalty: float = -1.0,
                illegal_bonus: float = 1.0) -> None:
    """Replay the duplicate match `duplicate_match` plays for these keys, pool and env_models (int32 [n, 2] by team or
    [n, 4] by player id) and, at every decision, play every legal alternative call out on that table with the nets' own
    argmax (DESIGN.md f16).  rewards_a / rewards_b (f32 [n, 4]) are the final Table_info rewards of that match.  Writes
    gain_sums int64 [M, 75, 38, 38, 4], regret_sums int64 [M, 75, 4], mismatch int64 [M], status int32[1] (_lib.MATCH_*) and,
    with `records`, one record per decision (records' env = env_offset + i), and with records made with `train=True` each
    record's training example (obs, gain; DESIGN.md f17).  Nothing is read back to the host."""
    n, M = int(keys.shape[0]), int(pool.shape[0]) if pool.dim() == 2 else 0
    if keys.dtype != torch.int64 or keys.dim() != 1:
        raise _lib.BrlError("call_values: keys must be int64 [n] (ops.make_keys)")
    _check_pool("call_values", pool, min_nets=1)
    _check_env_models("call_values", env_models, n)
    for name, t in (("rewards_a", rewards_a), ("rewards_b", rewards_b)):
        if t.dtype != torch.float32 or tuple(t.shape) != (n, 4):
            raise _lib.BrlError(f"call_values: {name} must be float32 [n, 4] (a Table_info's rewards)")
    _check_deal_table("call_values", table)
    if gain_sums.dtype != torch.int64 or tuple(gain_sums.shape) != (M,) + CALL_GAIN_SHAPE:
        raise _lib.BrlError(f"call_values: gain_sums must be int64 [{M}, 75, 38, 38, 4]")
    if regret_sums.dtype != torch.int64 or tuple(regret_sums.shape) != (M,) + CALL_REGRET_SHAPE:
        raise _lib.BrlError(f"call_values: regret_sums must be int64 [{M}, 75, 4]")
    if mismatch.dtype != torch.int64 or tuple(mismatch.shape) != (M,):
        raise _lib.BrlError(f"call_values: mismatch must be int64 [{M}]")
    if status.dtype != torch.int32 or status.numel() < 1:
        raise _lib.BrlError("call_values: status must be int32 [1]")
    if n and scratch.numel() < call_values_scratch_bytes(n, M):
        raise _lib.BrlError("call_values: scratch too small (ops.call_values_scratch_bytes)")
    if tune & F_SAMPLE:
        raise _lib.BrlError("call_values: sampling is not supported (argmax only)")
    if n and int(env_offset) < 0:
        raise _lib.BrlError("call_values: env_offset must be >= 0")
    flags = (F_MLP_BF16 if single_bf16 else 0) | (_lib.F_PLAYER_MODELS if env_models.shape[1] == 4 else 0) | tune
    _call("brl_call_values", [_ptr(keys), _ptr(table), _ptr(pool), _ptr(env_models), _ptr(rewards_a), _ptr(rewards_b),
                              _ptr(scratch), _ptr(gain_sums), _ptr(regret_sums), _ptr(mismatch), _ptr(status)]
          + (records.ptrs() if records is not None else [None] * 10),
          _params(n, k_steps=M, n_deals=table.shape[0], flags=flags, env_offset=env_offset,
                  seed=records.capacity if records is not None else 0, illegal_penalty=illegal_penalty,
                  illegal_bonus=illegal_bonus))


# ---- hand reading (DESIGN.md f18) -------------------------------------------------------------------------------------------
def hand_posterior_scratch_bytes(n_queries: int, n_samples: int, row_capacity: int, n_models: int) -> int:
    return _size_query("brl_hand_posterior_scratch_bytes", n_queries, n_samples, row_capacity, n_models)


def _check_posterior(who, table, calls, offsets, query, seat_nets, pool, scratch, outputs, *, N, row_capacity, board, dealer, vul,
                     temperature, path_flags, diagnostics, scratch_bytes):
    """the host checks of hand_posterior / hand_posterior_smc, in order; outputs and diagnostics: [(name, tensor, shape, dtype)]
    (the diagnostics all or none) -> Q, or None for an empty batch"""
    n = int(offsets.shape[0]) - 1 if offsets.dim() == 1 else -1
    Q = int(query.shape[0]) if query.dim() == 2 else -1
    if offsets.dtype != torch.int64 or n < 0:
        raise _lib.BrlError(f"{who}: offsets must be int64 [n + 1]")
    if calls.dtype != torch.uint8 or calls.dim() != 1:
        raise _lib.BrlError(f"{who}: calls must be u8 [total]")
    _check_deal_table(who, table)
    for name, t, dt in (("board", board, torch.int32), ("dealer", dealer, torch.int8), ("vul", vul, torch.uint8)):
        if t is not None and (t.dtype != dt or tuple(t.shape) != (n,)):
            raise _lib.BrlError(f"{who}: {name} must be {str(dt).replace('torch.', '')} [n]")
    if query.dtype != torch.int32 or tuple(query.shape) != (Q, 3):
        raise _lib.BrlError(f"{who}: query must be int32 [Q, 3] = (auction, observer seat, prefix length)")
    if seat_nets.dtype != torch.int32 or tuple(seat_nets.shape) != (Q, 4):
        raise _lib.BrlError(f"{who}: seat_nets must be int32 [Q, 4]")
    _check_pool(who, pool)
    M = int(pool.shape[0])
    if not 1 <= N <= 1 << 24:
        raise _lib.BrlError(f"{who}: samples must be in [1, 2^24]")
    if row_capacity < 0 or row_capacity % 256 or row_capacity > 1 << 30:
        raise _lib.BrlError(f"{who}: row_capacity must be a multiple of 256 in [0, 2^30]")
    if not (temperature >= 0.0) or temperature == float("inf"):
        raise _lib.BrlError(f"{who}: temperature must be finite and >= 0")
    if path_flags & ~(_lib.F_TUNE_MLP_LAYERS | _lib.F_TUNE_MLP_FUSED):
        raise _lib.BrlError(f"{who}: path_flags may hold F_TUNE_MLP_LAYERS / F_TUNE_MLP_FUSED only")
    for name, t, shape, dt in outputs(Q):
        if t.dtype != dt or tuple(t.shape) != shape:
            raise _lib.BrlError(f"{who}: {name} must be {str(dt).replace('torch.', '')} {list(shape)}")
    for group in diagnostics(Q):
        names = " and ".join(name for name, *_ in group)
        if len({t is None for _n, t, _s, _d in group}) > 1:
            raise _lib.BrlError(f"{who}: {names} go together")
        if group[0][1] is not None and any(t.dtype != dt or tuple(t.shape) != shape for _n, t, shape, dt in group):
            raise _lib.BrlError(f"{who}: " + ", ".join(f"{name} must be {str(dt).replace('torch.', '')} {list(shape)}"
                                                     for name, _t, shape, dt in group))
    if Q == 0:
        return None
    need = scratch_bytes(Q, N, row_capacity, M)
    if scratch.dtype != torch.uint8 or scratch.dim() != 1 or scratch.numel() < need:
        raise _lib.BrlError(f"{who}: scratch must be u8 [>= {need}] ({who}_scratch_bytes)")
    off, q, c = offsets.cpu(), query.cpu(), calls.cpu()
    if int(off[0]) != 0 or bool((off[1:] < off[:-1]).any()) or int(off[-1]) != calls.shape[0]:
        raise _lib.BrlError(f"{who}: offsets must rise from 0 to len(calls)")
    if c.numel() and int(c.max()) >= NUM_ACTIONS:
        raise _lib.BrlError(f"{who}: a call is outside 0..37")
    if int(q[:, 0].min()) < 0 or int(q[:, 0].max()) >= n:
        raise _lib.BrlError(f"{who}: a query's auction is outside [0, {n})")
    if board is None and n > table.shape[0]:
        raise _lib.BrlError(f"{who}: without board auction t needs deal row t: the table is too short")
    return Q


def _posterior_outputs(cards, features, weights, status):
    return lambda Q: (("cards", cards, (Q, 3, 52), torch.float64), ("features", features, (Q, 3, _lib.POST_FEATURES), torch.float64),
                      ("weights", weights, (Q, 4), torch.float64), ("status", status, (Q,), torch.int32))


def hand_posterior(table: torch.Tensor, calls: torch.Tensor, offsets: torch.Tensor, query: torch.Tensor, seat_nets: torch.Tensor,
                   pool: torch.Tensor, scratch: torch.Tensor, cards: torch.Tensor, features: torch.Tensor, weights: torch.Tensor,
                   status: torch.Tensor, *, samples: int, row_capacity: int, board: Optional[torch.Tensor] = None,
                   dealer: Optional[torch.Tensor] = None, vul: Optional[torch.Tensor] = None, seed: int = 0, query_offset: int = 0,
                   temperature: float = 1.0, single_bf16: bool = False, path_flags: int = 0, hands: Optional[torch.Tensor] = None,
                   logw: Optional[torch.Tensor] = None) -> None:
    """The posterior of the hidden hands for Q queries (brl_hand_posterior, DESIGN.md f18): query[j] = (t, s, L) reads the first L
    calls of auction t (calls[offsets[t]:offsets[t + 1]], u8 0..37, on deal row board[t] (None: row t), dealer dealer[t] (int8;
    None: North), vulnerability vul[t] (u8, bit 0 NS, bit 1 EW; None: none)) from absolute seat s, with net seat_nets[j, seat]
    (int32 [Q, 4]) of `pool` at each seat.  Writes cards f64[Q, 3, 52], features f64[Q, 3, 95], weights f64[Q, 4] and status
    int32[Q]; hands u64 (int64) [Q, N, 4] and logw f64[Q, N] are optional diagnostics, both or neither.  `row_capacity` (a
    multiple of 256) sizes the forward; the scratch is hand_posterior_scratch_bytes(Q, N, row_capacity, M) bytes.  Every
    argument is checked on the host (one device-to-host copy of offsets, calls and query) before any device work."""
    N = int(samples)
    Q = _check_posterior("hand_posterior", table, calls, offsets, query, seat_nets, pool, scratch,
                         _posterior_outputs(cards, features, weights, status), N=N, row_capacity=row_capacity, board=board,
                         dealer=dealer, vul=vul, temperature=temperature, path_flags=path_flags,
                         diagnostics=lambda Q: [[("hands", hands, (Q, N, 4), torch.int64), ("logw", logw, (Q, N), torch.float64)]],
                         scratch_bytes=hand_posterior_scratch_bytes)
    if Q is None:
        return
    flags = (F_MLP_BF16 if single_bf16 else 0) | int(path_flags)
    _call("brl_hand_posterior",
          [_ptr(table), _ptr(calls), _ptr(offsets), _ptr(board), _ptr(dealer), _ptr(vul), _ptr(query), _ptr(seat_nets), _ptr(pool),
           _ptr(scratch), _ptr(cards), _ptr(features), _ptr(weights), _ptr(status), _ptr(hands), _ptr(logw)],
          BrlParams(Q, int(query_offset), int(row_capacity), int(seed) & 0xFFFFFFFFFFFFFFFF, int(table.shape[0]), flags, N,
                    int(pool.shape[0]), -1.0, 1.0, float(temperature), 0.0))  # BrlParams directly: _params would turn a capacity of 0 into Q


# ---- hand reading by resample-move SMC (DESIGN.md f19) ----------------------------------------------------------------------
def hand_posterior_smc_scratch_bytes(n_queries: int, n_samples: int, row_capacity: int, n_models: int) -> int:
    return _size_query("brl_hand_posterior_smc_scratch_bytes", n_queries, n_samples, row_capacity, n_models)


SMC_TRACE = ("loglik", "ancestors", "pairs", "accepted", "proposed")


def smc_trace(Q: int, N: int, stages: int, moves: int, device) -> dict:
    """empty trace buffers of brl_hand_posterior_smc: loglik f64[Q, K, N], ancestors i32[Q, K, N], pairs i32[Q, K, R],
    accepted u8[Q, K, R, N], proposed f64[Q, K, R, N, 2]"""
    K, R = int(stages), int(moves)
    return dict(loglik=torch.empty((Q, K, N), dtype=torch.float64, device=device),
                ancestors=torch.empty((Q, K, N), dtype=torch.int32, device=device),
                pairs=torch.empty((Q, K, R), dtype=torch.int32, device=device),
                accepted=torch.empty((Q, K, R, N), dtype=torch.uint8, device=device),
                proposed=torch.empty((Q, K, R, N, 2), dtype=torch.float64, device=device))


def hand_posterior_smc(table: torch.Tensor, calls: torch.Tensor, offsets: torch.Tensor, query: torch.Tensor, seat_nets: torch.Tensor,
                       pool: torch.Tensor, scratch: torch.Tensor, cards: torch.Tensor, features: torch.Tensor, weights: torch.Tensor,
                       status: torch.Tensor, log_evidence: torch.Tensor, resamples: torch.Tensor, acceptance: torch.Tensor, *,
                       samples: int, row_capacity: int, stages: int, moves: int = 1, ess_threshold: float = 0.5,
                       board: Optional[torch.Tensor] = None, dealer: Optional[torch.Tensor] = None,
                       vul: Optional[torch.Tensor] = None, seed: int = 0, query_offset: int = 0, temperature: float = 1.0,
                       single_bf16: bool = False, path_flags: int = 0, hands: Optional[torch.Tensor] = None,
                       logw: Optional[torch.Tensor] = None, ell: Optional[torch.Tensor] = None,
                       trace: Optional[dict] = None) -> None:
    """The posterior of hand_posterior by resample-move SMC over the calls of each prefix (brl_hand_posterior_smc, DESIGN.md
    f19).  Arguments and outputs as hand_posterior, plus log_evidence f64[Q], resamples int32[Q] and acceptance f64[Q];
    `stages` >= every query's L (a longer prefix gets POST_STAGES), `moves` in [0, 64] Metropolis-Hastings moves after each
    resample, `ess_threshold` kappa in [0, 1] (resample when ESS < kappa N; 1 resamples at every stage).  `row_capacity`
    bounds each stage's and each move's forward.  Optional: hands / logw / ell f64[Q, N, 3] (the final particles, all or
    none) and `trace` (smc_trace's five buffers, all or none).  Every argument is checked before any device work."""
    who, N, K, R = "hand_posterior_smc", int(samples), int(stages), int(moves)
    if not 0 <= R <= _lib.SMC_MAX_MOVES:
        raise _lib.BrlError(f"{who}: moves must be in [0, {_lib.SMC_MAX_MOVES}]")
    if not 0 <= K <= _lib.SMC_MAX_STAGES:
        raise _lib.BrlError(f"{who}: stages must be in [0, {_lib.SMC_MAX_STAGES}]")
    if not 0.0 <= ess_threshold <= 1.0:
        raise _lib.BrlError(f"{who}: ess_threshold must be in [0, 1]")
    tr = trace or {}
    if trace is not None and set(trace) != set(SMC_TRACE):
        raise _lib.BrlError(f"{who}: trace must hold {', '.join(SMC_TRACE)}")
    base = _posterior_outputs(cards, features, weights, status)
    outputs = lambda Q: base(Q) + (("log_evidence", log_evidence, (Q,), torch.float64), ("resamples", resamples, (Q,), torch.int32),  # noqa: E731
                                   ("acceptance", acceptance, (Q,), torch.float64))
    diagnostics = lambda Q: [  # noqa: E731
        [("hands", hands, (Q, N, 4), torch.int64), ("logw", logw, (Q, N), torch.float64), ("ell", ell, (Q, N, 3), torch.float64)],
        [("trace loglik", tr.get("loglik"), (Q, K, N), torch.float64), ("trace ancestors", tr.get("ancestors"), (Q, K, N), torch.int32),
         ("trace pairs", tr.get("pairs"), (Q, K, R), torch.int32), ("trace accepted", tr.get("accepted"), (Q, K, R, N), torch.uint8),
         ("trace proposed", tr.get("proposed"), (Q, K, R, N, 2), torch.float64)]]
    Q = _check_posterior(who, table, calls, offsets, query, seat_nets, pool, scratch, outputs, N=N, row_capacity=row_capacity,
                         board=board, dealer=dealer, vul=vul, temperature=temperature, path_flags=path_flags,
                         diagnostics=diagnostics, scratch_bytes=hand_posterior_smc_scratch_bytes)
    if Q is None:
        return
    flags = (F_MLP_BF16 if single_bf16 else 0) | int(path_flags)
    post = BrlParams(Q, int(query_offset), int(row_capacity), int(seed) & 0xFFFFFFFFFFFFFFFF, int(table.shape[0]), flags, N,
                     int(pool.shape[0]), -1.0, 1.0, float(temperature), 0.0)
    _call("brl_hand_posterior_smc",
          [_ptr(table), _ptr(calls), _ptr(offsets), _ptr(board), _ptr(dealer), _ptr(vul), _ptr(query), _ptr(seat_nets), _ptr(pool),
           _ptr(scratch), _ptr(cards), _ptr(features), _ptr(weights), _ptr(status), _ptr(log_evidence), _ptr(resamples),
           _ptr(acceptance), _ptr(hands), _ptr(logw), _ptr(ell)] + [_ptr(tr.get(k)) for k in SMC_TRACE],
          _lib.BrlSmcParams(post, float(ess_threshold), R, K, 0))
