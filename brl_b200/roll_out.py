"""`make_roll_out` of src/roll_out.py:23-110: T env steps of the learner against an
opponent net through the auto-reset quad step, recording `Transition`s.

Buffers: the trajectory is preallocated [T, N, ...] and the kernels write into it in place -- the env kernel of step t
writes the observation / mask that step t+1 records straight into slot t+1 (in the policy's input dtype, bf16), the quad
step's OR-ed `terminated` straight into `done[t]`, and the player to act into one of two alternating buffers, so the
"actor" of step t is still there when `rewards[actor]` is taken; `terminated_count` is accumulated by that same kernel.
One rollout step is 13 launches (4 policy forwards, each a counter memset + one persistent kernel; 4 env steps; the reward
gather) and nothing else.

CUDA graph: every op is enqueue-only, so from 4096 envs on (the fused-forward size) the whole T-step rollout is captured
ONCE per (shape, opponent) into a CUDA graph and replayed: parameters are re-packed into fixed-address blobs before a
replay (an opponent given as models.PackedParams, e.g. from zoo.ModelZoo, is copied device to device), the env state / last observation are copied into the graph's own buffers (device-to-device memcpy), and the
per-rollout PRNG key is a device word XORed into every captured sampling seed (BRL_F_SEED_SALT).  The returned
trajectory then aliases the graph's buffers: it is valid until the next call of the same roll_out.
`BRL_ROLLOUT_GRAPH=0` (or `trace=`) selects the plain launch path.

Anchor (a KL-anchored PPO run, ppo.py `anchor_model_path`): `roll_out(runner_state, opp_params, anchor_params)` also runs
the anchor net on every step's observation (one `brl_mlp_forward` on the same bf16 `obs[t]`) into f32
`roll_out.anchor_logits[T, n, 38]`, which the update's KL term reads.  The buffer belongs to the roll-out and, like the
trajectory, stays valid until the next call.  Anchored and plain calls keep separate buffers and CUDA graphs; the anchor
is packed into its own fixed-address blob before an anchored replay.

Partner (ppo.py `partner_model_path`): `roll_out(runner_state, opp_params, partner_params=...)` plays the quad step's
sub-step 3 -- the actor's partner slot -- with that net instead of the actor (utils._QuadStep; sampled, not recorded).  That
forward runs anyway, so a partner costs one more blob pack per graph replay: partnered calls keep their own buffers and
CUDA graph, with the partner packed into its own fixed-address blob.

Reward (config["reward_mode"]): "score" (the default) is the reference's rewards[actor] / reward_scale.  "par_imp" takes a
finished board's reward against its double-dummy par (DESIGN.md f13) instead: IMP(rewards[actor] - par[actor]) / 24.  Before
each quad step `brl_par` writes the par of the state in `buf.packed` into the rollout's `par[n, 4]`: that state still holds
the deal the quad step may finish, since auto-reset happens inside the step.  After the step `brl_gather_reward_par` replaces
the reward gather.  Par mode is for competitive games with masked actors only (check_reward_mode).
"""
from __future__ import annotations

import os
from typing import NamedTuple

import torch

from . import ops
from . import random as brandom
from .env import State
from .utils import WithOutputs, auto_reset, single_play_step_free_run, single_play_step_two_policy_commpetitive

_GRAPH_MIN_ENVS = 4096  # BRL_F_SEED_SALT lives in the fused forward launch
_CAPTURE_KEY = 0x5EED    # host key the captured seeds are split from; the per-rollout key is the device salt
REWARD_MODES = ("score", "par_imp")


def check_reward_mode(config) -> None:
    """ValueError for an unknown config["reward_mode"], and for "par_imp" in free-run games (the opponents never bid, so
    competitive par is the wrong baseline) or without actor_illegal_action_mask (an illegal call ends a board with a
    penalty, not a contract score)."""
    mode = config.get("reward_mode", "score")
    if mode not in REWARD_MODES:
        raise ValueError(f"reward_mode must be one of {REWARD_MODES}; got {mode!r}")
    if mode == "par_imp":
        if config["game_mode"] == "free-run":
            raise ValueError('reward_mode="par_imp" needs game_mode="competitive": in free-run the opponents never bid')
        if not config["actor_illegal_action_mask"]:
            raise ValueError('reward_mode="par_imp" needs actor_illegal_action_mask: an illegal call ends a board with a '
                             'penalty, not a contract score')


class Transition(NamedTuple):
    """src/roll_out.py:13-20"""
    done: torch.Tensor
    action: torch.Tensor
    value: torch.Tensor
    reward: torch.Tensor
    log_prob: torch.Tensor
    obs: torch.Tensor
    legal_action_mask: torch.Tensor


class _Buffers:
    """Everything one rollout reads and writes, at fixed addresses."""

    def __init__(self, T, n, dev, obs_dtype, par_mode=False):
        self.T, self.n = T, n
        self.done = torch.empty((T, n), dtype=torch.uint8, device=dev)
        self.action = torch.empty((T, n), dtype=torch.int32, device=dev)
        self.value = torch.empty((T, n), dtype=torch.float32, device=dev)
        self.reward = torch.empty((T, n), dtype=torch.float32, device=dev)
        self.log_prob = torch.empty((T, n), dtype=torch.float32, device=dev)
        self.obs = torch.empty((T + 1, n, ops.OBS_DIM), dtype=obs_dtype, device=dev)       # slot T = the next rollout's slot 0
        self.mask = torch.empty((T + 1, n, ops.NUM_ACTIONS), dtype=torch.uint8, device=dev)
        self.packed = ops.new_state(n, dev)
        self.rewards = torch.empty((n, 4), dtype=torch.float32, device=dev)
        self.player = torch.empty((2, n), dtype=torch.int8, device=dev)                    # player to act, alternating per step
        self.term0 = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.count = torch.zeros(1, dtype=torch.int64, device=dev)
        self.par = torch.empty((n, 4), dtype=torch.float32, device=dev) if par_mode else None  # par of the pre-step state

    def state(self, env, t):
        """State view whose outputs are the buffers step t writes (obs / mask slot t, done[t-1], player[t % 2])"""
        out = ops.EnvOutputs.__new__(ops.EnvOutputs)
        out.observation, out.legal_action_mask, out.rewards = self.obs[t], self.mask[t], self.rewards
        out.terminated = self.done[t - 1] if t > 0 else self.term0
        out.current_player = self.player[t % 2]
        return State(env, self.packed, out)

    def load(self, env_state, last_obs):
        """copy the caller's env state in (device-to-device copies; a cast launch only if the observation dtype differs)"""
        if env_state._packed.data_ptr() != self.packed.data_ptr():
            self.packed.copy_(env_state._packed)
        if last_obs.dtype == self.obs.dtype:
            if last_obs.data_ptr() != self.obs[0].data_ptr():
                self.obs[0].copy_(last_obs)
        else:
            ops.obs_to_bf16(last_obs.contiguous(), out=self.obs[0])
        if env_state._mask_u8.data_ptr() != self.mask[0].data_ptr():
            self.mask[0].copy_(env_state._mask_u8)
        if env_state.current_player.data_ptr() != self.player[0].data_ptr():
            self.player[0].copy_(env_state.current_player)


def make_roll_out(config, env, actor_forward_pass, opp_forward_pass, anchor_forward_pass=None, partner_forward_pass=None):
    masked = bool(config["actor_illegal_action_mask"])
    if not masked and not config.get("actor_illegal_action_penalty", False):
        raise ValueError("one of actor_illegal_action_mask / actor_illegal_action_penalty must be set (src/roll_out.py:24-39)")
    if config["game_mode"] == "competitive":
        make_step_fn = single_play_step_two_policy_commpetitive
    elif config["game_mode"] == "free-run":
        make_step_fn = single_play_step_free_run
    else:
        raise ValueError(config["game_mode"])
    check_reward_mode(config)
    reward_mode = config.get("reward_mode", "score")
    par_mode = reward_mode == "par_imp"
    T = int(config["num_steps"])
    scale = float(config["reward_scale"])
    obs_dtype = getattr(actor_forward_pass, "input_dtype", torch.float32)
    cache = {}  # (n, anchored, reward_mode, partnered) -> dict(buf, graph, blobs, salt, anchor_logits, ...)
    out = {"anchor_logits": None}

    def body(buf, params, opp_params, rng, trace, anchor=None, partner_params=None):
        """the T steps of src/roll_out.py:49-108 on `buf`"""
        step_fn = make_step_fn(step_fn=auto_reset(env.step, env.init), actor_forward_pass=actor_forward_pass,
                               actor_params=params, opp_forward_pass=opp_forward_pass, opp_params=opp_params,
                               partner_forward_pass=partner_forward_pass if partner_params is not None else None,
                               partner_params=partner_params)
        step_fn.trace = trace
        cur = buf.state(env, 0)
        for t in range(T):
            rng, _rng = brandom.split(rng)
            actor_forward_pass.act(params, buf.obs[t], buf.mask[t] if masked else None, buf.action[t], buf.log_prob[t],
                                   buf.value[t], sample=True, seed=_rng, env_offset=getattr(env, "env_offset", 0))  # :73-81
            if anchor is not None:  # the anchor's logits on the observation the actor just saw
                anchor_params, anchor_logits, anchor_value = anchor
                anchor_forward_pass.forward_into(anchor_params, buf.obs[t], anchor_logits[t], anchor_value)
            rng, _rng = brandom.split(rng)
            if par_mode:
                ops.par(buf.packed, env.table, buf.par)
            cur = step_fn(cur, buf.action[t], _rng, out_state=buf.state(env, t + 1))                                # :84
            # reward = rewards[actor] / scale with actor = the player who was to act BEFORE the quad step (still in the
            # other player buffer), and terminated_count += sum(done)                                             :85-94
            if par_mode:
                ops.gather_reward_par(buf.rewards, buf.player[t % 2], buf.par, buf.done[t], buf.reward[t], count=buf.count)
            else:
                ops.gather_reward(buf.rewards, buf.player[t % 2], buf.reward[t], scale, done=buf.done[t], count=buf.count)
        return cur, rng

    def finish(buf, params, opt_state, cur, terminated_count, rng):
        total = terminated_count + buf.count[0]
        traj = Transition(done=buf.done.view(torch.bool), action=buf.action, value=buf.value, reward=buf.reward,
                          log_prob=buf.log_prob, obs=buf.obs[:T], legal_action_mask=buf.mask[:T].view(torch.bool))
        return (params, opt_state, cur, cur.observation, total, rng), traj

    def roll_out(runner_state, opp_params, anchor_params=None, partner_params=None, trace=None, graph_seeding=False):
        """`anchor_params`: also record the anchor net's logits of every step in `roll_out.anchor_logits` (needs
        `anchor_forward_pass`).  `partner_params`: the net of the quad step's sub-step 3 instead of the actor (needs
        `partner_forward_pass`).  `trace` (tests): a list that receives every sub-step action tensor; forces the plain
        launch path.  `graph_seeding` (tests): plain launches with exactly the seeds a graph replay uses (captured constants
        XOR the per-rollout salt), so that a graph replay can be compared bit for bit with a traced, oracle-checked run."""
        params, opt_state, env_state, last_obs, terminated_count, rng = runner_state
        n, dev = env_state.num_envs, env.device
        anchored = anchor_params is not None
        if anchored and anchor_forward_pass is None:
            raise ValueError("roll_out got anchor_params, but make_roll_out was given no anchor_forward_pass")
        partnered = partner_params is not None
        if partnered and partner_forward_pass is None:
            raise ValueError("roll_out got partner_params, but make_roll_out was given no partner_forward_pass")
        use_graph = trace is None and not graph_seeding and n >= _GRAPH_MIN_ENVS and \
            os.environ.get("BRL_ROLLOUT_GRAPH", "1") != "0" and \
            hasattr(actor_forward_pass, "pack_into") and hasattr(opp_forward_pass, "pack_into") and \
            (not anchored or hasattr(anchor_forward_pass, "pack_into")) and \
            (not partnered or hasattr(partner_forward_pass, "pack_into"))  # tensor-core nets only
        # the forward passes whose sampling seeds take the per-rollout salt
        salted = (actor_forward_pass, opp_forward_pass) + ((partner_forward_pass,) if partnered else ())
        c = cache.get((n, anchored, reward_mode, partnered))
        if c is None:
            c = cache[(n, anchored, reward_mode, partnered)] = {"buf": _Buffers(T, n, dev, obs_dtype, par_mode), "graph": None}
            if anchored:
                c["anchor_logits"] = torch.empty((T, n, ops.NUM_ACTIONS), dtype=torch.float32, device=dev)
                c["anchor_value"] = torch.empty(n, dtype=torch.float32, device=dev)
        out["anchor_logits"] = c["anchor_logits"] if anchored else None
        buf = c["buf"]
        buf.load(env_state, last_obs)
        buf.count.zero_()
        if not use_graph:
            prev = [getattr(fp, "seed_salt", None) for fp in salted]
            salt, body_rng = None, rng
            if graph_seeding:
                rng, key = brandom.split(rng)
                salt = torch.tensor([key - (1 << 64) if key >= (1 << 63) else key], dtype=torch.int64, device=dev)
                body_rng = _CAPTURE_KEY
            for fp in salted:
                fp.seed_salt = salt
            anchor = (anchor_params, c["anchor_logits"], c["anchor_value"]) if anchored else None
            try:
                cur, body_rng = body(buf, params, opp_params, body_rng, trace, anchor, partner_params)
            finally:
                for fp, v in zip(reversed(salted), reversed(prev)):  # restored in reverse: a pass listed twice ends as it was
                    fp.seed_salt = v
            return finish(buf, params, opt_state, cur, terminated_count, rng if graph_seeding else body_rng)
        # ---- CUDA-graph path ----
        if c["graph"] is None:
            c["salt"] = torch.zeros(1, dtype=torch.int64, device=dev)
            c["salt_host"] = torch.zeros(1, dtype=torch.int64).pin_memory()
            c["blobs"] = (torch.empty(ops._lib.load().brl_mlp_packed_bytes(), dtype=torch.uint8, device=dev),
                          torch.empty(ops._lib.load().brl_mlp_packed_bytes(), dtype=torch.uint8, device=dev))
        rng, key = brandom.split(rng)
        c["salt_host"][0] = key - (1 << 64) if key >= (1 << 63) else key
        c["salt"].copy_(c["salt_host"], non_blocking=True)
        fixed_a, fixed_o = {"_brl_packed_fixed": c["blobs"][0]}, {"_brl_packed_fixed": c["blobs"][1]}
        actor_forward_pass.pack_into(params, c["blobs"][0])
        (opp_forward_pass if opp_params is not params else actor_forward_pass).pack_into(opp_params, c["blobs"][1])
        anchor = None
        if anchored:
            if "anchor_blob" not in c:
                c["anchor_blob"] = torch.empty(ops._lib.load().brl_mlp_packed_bytes(), dtype=torch.uint8, device=dev)
            anchor_forward_pass.pack_into(anchor_params, c["anchor_blob"])
            anchor = ({"_brl_packed_fixed": c["anchor_blob"]}, c["anchor_logits"], c["anchor_value"])
        partner = None
        if partnered:
            if "partner_blob" not in c:
                c["partner_blob"] = torch.empty(ops._lib.load().brl_mlp_packed_bytes(), dtype=torch.uint8, device=dev)
            partner_forward_pass.pack_into(partner_params, c["partner_blob"])
            partner = {"_brl_packed_fixed": c["partner_blob"]}
        if c["graph"] is None:
            prev = [getattr(fp, "seed_salt", None) for fp in salted]
            for fp in salted:
                fp.seed_salt = c["salt"]  # baked into the captured launches only
            saved = (buf.packed.clone(), buf.obs[0].clone(), buf.mask[0].clone(), buf.player[0].clone())
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            try:
                with torch.cuda.stream(side):
                    body(buf, fixed_a, fixed_o, _CAPTURE_KEY, None, anchor, partner)  # warm-up: lazy allocations (scratch), attribute calls
                    buf.packed.copy_(saved[0]); buf.obs[0].copy_(saved[1]); buf.mask[0].copy_(saved[2]); buf.player[0].copy_(saved[3])
                    buf.count.zero_()
                    side.synchronize()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=side):
                        body(buf, fixed_a, fixed_o, _CAPTURE_KEY, None, anchor, partner)
            finally:
                for fp, v in zip(reversed(salted), reversed(prev)):
                    fp.seed_salt = v
            torch.cuda.current_stream(dev).wait_stream(side)
            c["graph"] = g
            buf.packed.copy_(saved[0]); buf.obs[0].copy_(saved[1]); buf.mask[0].copy_(saved[2]); buf.player[0].copy_(saved[3])
            buf.count.zero_()
        c["graph"].replay()
        cur = buf.state(env, T)
        return finish(buf, params, opt_state, cur, terminated_count, rng)

    return WithOutputs(roll_out, out)
