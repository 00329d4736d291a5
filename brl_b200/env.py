"""pgx-1.4.0-shaped `bridge_bidding` Env surface over the CUDA C ABI.

This is the host-side mirror of the interface brl consumes (SURVEY 8b):
`BridgeBidding(dds_path)`, `env.init(key)`, `env.step(state, action)`,
`env.observation_shape`, and a `State` with `current_player`, `observation`,
`legal_action_mask`, `rewards`, `terminated`, `truncated` plus the private fields
brl reads (`_last_bid`, `_last_bidder`, `_call_x`, `_call_xx`, `_dealer`,
`_shuffled_players`, `_vul_NS`, `_vul_EW`, `_pass_num`, `_step_count`, `_rng_key`).
Reference call sites: eval.py:43, src/evaluation.py:92-112, src/roll_out.py:51,72-100,
src/duplicate.py:6,120-135,149, src/utils.py:36-53, ppo.py:241,305.

Differences a porter must know (documented, not hidden):
  * natively batched: every tensor has a leading env axis N; the reference's
    `jax.vmap(env.step)` folds into N (no per-env calls);
  * state lives in HBM as 80 B/env of packed words (`State._packed`); private
    fields are unpacked on demand by a kernel (`brl_state_fields`);
  * keys are 64-bit counter-based (Philox) keys as int64 tensors, not threefry
    `uint32[2]` -- which deal/dealer/vul/seating a key maps to is a pgx-internal
    convention nothing in the tree pins (parity is conditional on the same draws);
  * there is no CPU path: tensors must be CUDA tensors.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import deals as _deals
from . import ops


class State:
    """Batched env state.  Public tensors are the buffers the kernels wrote."""

    __slots__ = ("env", "_packed", "observation", "_mask_u8", "rewards", "_terminated_u8", "current_player", "_fields")

    def __init__(self, env, packed, out: ops.EnvOutputs):
        self.env = env
        self._packed = packed
        self.observation = out.observation
        self._mask_u8 = out.legal_action_mask
        self.rewards = out.rewards
        self._terminated_u8 = out.terminated
        self.current_player = out.current_player
        self._fields = None

    # -- pgx public fields -------------------------------------------------
    @property
    def legal_action_mask(self) -> torch.Tensor:
        return self._mask_u8.view(torch.bool)

    @property
    def terminated(self) -> torch.Tensor:
        return self._terminated_u8.view(torch.bool)

    @property
    def truncated(self) -> torch.Tensor:
        return torch.zeros_like(self._terminated_u8).view(torch.bool)  # bridge bidding never truncates

    @property
    def num_envs(self) -> int:
        return self._packed.shape[1]

    def outputs(self) -> ops.EnvOutputs:
        o = ops.EnvOutputs.__new__(ops.EnvOutputs)
        o.observation, o.legal_action_mask, o.rewards = self.observation, self._mask_u8, self.rewards
        o.terminated, o.current_player = self._terminated_u8, self.current_player
        return o

    # -- pgx private fields brl reads ----------------------------------------
    def _f(self, name):
        if self._fields is None:
            self._fields = ops.state_fields(self._packed)
        return self._fields[name]

    _step_count = property(lambda s: s._f("step_count"))
    _rng_key = property(lambda s: s._f("rng_key"))
    _shuffled_players = property(lambda s: s._f("shuffled_players"))
    _dealer = property(lambda s: s._f("dealer"))
    _vul_NS = property(lambda s: s._f("vul")[:, 0].view(torch.bool))
    _vul_EW = property(lambda s: s._f("vul")[:, 1].view(torch.bool))
    _last_bid = property(lambda s: s._f("last_bid"))
    _last_bidder = property(lambda s: s._f("last_bidder"))
    _call_x = property(lambda s: s._f("call_x").view(torch.bool))
    _call_xx = property(lambda s: s._f("call_xx").view(torch.bool))
    _pass_num = property(lambda s: s._f("pass_num"))
    _deal = property(lambda s: s._f("deal"))

    def replace(self, **kw) -> "State":
        """`state.replace(...)` for the Env-surface tensors (src/duplicate.py:135,159-162).
        Packed private fields are rewritten by kernels (reset_fields / duplicate_init), not here."""
        new = State.__new__(State)
        for k in State.__slots__:
            setattr(new, k, getattr(self, k))
        for k, v in kw.items():
            if k == "rewards":
                new.rewards = v
            elif k == "observation":
                new.observation = v
            elif k == "legal_action_mask":
                new._mask_u8 = v.view(torch.uint8)
            elif k == "current_player":
                new.current_player = v
            else:
                raise NotImplementedError(f"State.replace({k}=...) is not supported; use the env ops that rewrite the packed state")
        return new


class BridgeBidding:
    """Drop-in for `pgx.bridge_bidding.BridgeBidding` (eval.py:43, ppo.py:233,252,303)."""

    id = "bridge_bidding"
    version = "brl-b200"
    num_players = 4
    num_actions = ops.NUM_ACTIONS
    observation_shape = (ops.OBS_DIM,)

    def __init__(self, dds_results_table_path: Optional[str] = None, *, table: Optional[np.ndarray] = None,
                 device="cuda", obs_dtype=torch.float32, illegal_action_penalty: float = -1.0,
                 illegal_action_bonus: float = 1.0, synthetic_deals: int = 100_000, seed: int = 0,
                 env_offset: int = 0):
        if table is None:
            if dds_results_table_path is not None:
                table = _deals.load_table(dds_results_table_path)
            else:  # the DDS dataset cannot be downloaded offline (README.md:11-15): synthetic table
                table = _deals.synthetic_deal_table(synthetic_deals, seed=seed)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("brl_b200.BridgeBidding needs a CUDA device (there is no CPU path)")
        self.table_np = np.ascontiguousarray(table, dtype=np.uint8).reshape(-1, _deals.DEAL_ROW_BYTES)
        self.table = torch.as_tensor(self.table_np, device=self.device)
        self.n_deals = self.table.shape[0]
        self.obs_dtype = obs_dtype
        self.illegal_penalty = float(illegal_action_penalty)
        self.illegal_bonus = float(illegal_action_bonus)
        self.env_offset = int(env_offset)  # global index of this rank's env 0 (sharding, SURVEY 8e)

    # -- allocation helpers -------------------------------------------------
    def _fresh(self, n: int):
        return ops.new_state(n, self.device), ops.EnvOutputs(n, self.device, self.obs_dtype)

    def make_keys(self, seed: int, n: int, env_offset: int = 0) -> torch.Tensor:
        """`jax.random.split(key, n)` analogue (src/evaluation.py:93-94): one key per GLOBAL env index."""
        return ops.make_keys(seed, n, self.device, env_offset)

    # -- Env API ----------------------------------------------------------------
    def init(self, key: torch.Tensor) -> State:
        """`jax.vmap(env.init)(keys)` (src/evaluation.py:95)."""
        packed, out = self._fresh(key.shape[0])
        ops.init(key, self.table, packed, out)
        return State(self, packed, out)

    def init_from(self, deal, dealer, vul_ns, vul_ew, shuffled_players, rng_key=None) -> State:
        """Start episodes on GIVEN draws (what `State(...)`/`replace` construction does in
        src/duplicate.py:120-128; also how parity tests share draws with the oracle)."""
        dev = self.device
        t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dt).contiguous()  # noqa: E731
        deal_t = t(deal, torch.int32)
        packed, out = self._fresh(deal_t.shape[0])
        ops.reset_fields(deal_t, t(dealer, torch.int32), t(vul_ns, torch.uint8), t(vul_ew, torch.uint8),
                         t(shuffled_players, torch.int8), None if rng_key is None else t(rng_key, torch.int64),
                         self.table, packed, out)
        return State(self, packed, out)

    def step(self, state: State, action: torch.Tensor, *, inplace: bool = False, autoreset: bool = False) -> State:
        """`jax.vmap(env.step)(state, action)` (src/roll_out.py:51, src/duplicate.py:149).
        Functional by default (new buffers); `inplace=True` aliases state and outputs."""
        n = state.num_envs
        if inplace:
            packed, out = state._packed, state.outputs()
        else:
            packed, out = self._fresh(n)
        ops.step(state._packed, action.to(torch.int32), self.table, packed, out, autoreset=autoreset,
                 illegal_penalty=self.illegal_penalty, illegal_bonus=self.illegal_bonus)
        return State(self, packed, out)

    def observe(self, state: State, player_id: Optional[torch.Tensor] = None) -> torch.Tensor:
        """`_observe(state, player)` (src/duplicate.py:6,134)."""
        odt = torch.uint8 if self.obs_dtype == torch.bool else self.obs_dtype
        obs = torch.empty((state.num_envs, ops.OBS_DIM), dtype=odt, device=self.device)
        ops.observe(state._packed, self.table, obs, None if player_id is None else player_id.to(torch.int8))
        return obs

    def par(self, state: State):
        """Double-dummy par of each env's board (DESIGN.md f13) -> (par f32[n, 4] by player id, as `rewards` is laid out,
        contract i32[n]: -1 passed out, else bid | declarer_seat << 8 | doubled << 10)."""
        n = state.num_envs
        par = torch.empty((n, 4), dtype=torch.float32, device=self.device)
        contract = torch.empty(n, dtype=torch.int32, device=self.device)
        ops.par(state._packed, self.table, par, contract)
        return par, contract


def act_randomly(seed: int, state: State, step_index: int = 0, env_offset: int = 0) -> torch.Tensor:
    """`pgx.experimental.utils.act_randomly(key, state)` (src/duplicate.py:7,234): a uniform
    random LEGAL action per env, drawn by the same counter-based rule the fused rollout uses."""
    n = state.num_envs
    logits = torch.zeros((n, ops.NUM_ACTIONS), dtype=torch.float32, device=state._packed.device)
    action = torch.empty(n, dtype=torch.int32, device=logits.device)
    ops.categorical(logits, state._mask_u8, action, None, sample=True, seed=seed, env_offset=env_offset,
                    step_index=step_index)
    return action
