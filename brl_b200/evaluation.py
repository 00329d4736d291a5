"""Evaluation loops of src/evaluation.py: `make_simple_duplicate_evaluate` (69-204, the
eval.py path and the league probe), `make_simple_evaluate` (11-66) and `make_evaluate` (207-1032),
each as a host loop and as a device loop (one brl_duplicate_match / brl_evaluate_match call)."""
from __future__ import annotations

import torch

from . import dist as bdist
from . import ops
from . import random as brandom
from .duplicate import Table_info, duplicate_step
from .models import load_params, make_forward_pass
from .utils import single_play_step_two_policy_commpetitive_deterministic

_CHECK_EVERY = 8  # stepping a finished env is a zero-reward no-op, so the all-done test needs no per-step sync


class _TeamRows:
    """Per-iteration lists of the envs still playing, split by the team of the player to act (brl_team_rows).  The
    reference's vmapped loop (src/evaluation.py:124-151) runs BOTH nets on every env and keeps forwarding finished envs
    until the slowest auction ends; here each net runs on exactly the envs it decides.  The two counts come back to the
    host once per iteration (8 bytes): they size the two forward launches and are the loop's termination test."""

    def __init__(self, n: int, device):
        self.rows1 = torch.empty(n, dtype=torch.int32, device=device)
        self.rows2 = torch.empty(n, dtype=torch.int32, device=device)
        self.counts = torch.zeros(2, dtype=torch.int32, device=device)
        self.host = torch.zeros(2, dtype=torch.int32).pin_memory()
        self.forwarded = 0  # rows sent through a net so far (tests / bench: compare with iterations * 2 * n)

    def split(self, current_player, done_u8):
        ops.team_rows(current_player, done_u8, self.rows1, self.rows2, self.counts)
        self.host.copy_(self.counts, non_blocking=True)
        torch.cuda.current_stream(self.counts.device).synchronize()
        c1, c2 = int(self.host[0]), int(self.host[1])
        self.forwarded += c1 + c2
        return self.rows1[:c1], self.rows2[:c2]


def _act_team(forward_pass, params, partner, state, action, rows, logits=None):
    """the team of `rows` decides: `params` for all of them, or, with a `partner`, `params` for the team's first player
    (player id 0 / 2) and `partner` for the second (1 / 3)"""
    if partner is None:
        forward_pass.act_rows(params, state.observation, state._mask_u8, action, rows, logits=logits)
        return
    second = (state.current_player[rows.long()] & 1).bool()
    forward_pass.act_rows(params, state.observation, state._mask_u8, action, rows[~second], logits=logits)
    forward_pass.act_rows(partner, state.observation, state._mask_u8, action, rows[second], logits=logits)


def _bf16_state(env, keys):
    """env.init with the observation written directly in bf16 (the tensor-core nets' input dtype; the observation of
    these loops is read by the nets only)"""
    n = keys.shape[0]
    from .env import State
    packed, out = ops.new_state(n, env.device), ops.EnvOutputs(n, env.device, torch.bfloat16)
    ops.init(keys, env.table, packed, out)
    return State(env, packed, out)


def _opponent_params(eval_env, team2_params, team2_model_path, game_mode: str = "competitive"):
    """team 2's net: `team2_params`, else the pickle at `team2_model_path`; None in "free-run" (team 2 always passes)"""
    if game_mode == "competitive":
        return team2_params if team2_params is not None else load_params(team2_model_path, eval_env.device)
    if game_mode == "free-run":
        return None
    raise ValueError(game_mode)


def make_simple_evaluate(eval_env, team1_activation, team1_model_type, team2_activation, team2_model_type,
                         team2_model_path, num_eval_envs, team2_params=None):
    """src/evaluation.py:11-66: deterministic quad steps vs a fixed opponent; mean raw score."""
    actor_forward_pass = make_forward_pass(activation=team1_activation, model_type=team1_model_type)
    opp_forward_pass = make_forward_pass(activation=team2_activation, model_type=team2_model_type)
    opp_params = _opponent_params(eval_env, team2_params, team2_model_path)

    def simple_evaluate(actor_params, rng, trace=None, partner_params=None):
        """`trace` (a list, tests only) receives the four sub-step action tensors of every quad step and finally
        ("R", per-env return) -- the inputs of an oracle replay.  `partner_params`: the actor's partner (the quad step's
        sub-step 3, of the actor's architecture) instead of the actor itself."""
        step_fn = single_play_step_two_policy_commpetitive_deterministic(
            step_fn=eval_env.step, actor_params=actor_params, actor_forward_pass=actor_forward_pass,
            opp_params=opp_params, opp_forward_pass=opp_forward_pass,
            partner_forward_pass=actor_forward_pass if partner_params is not None else None, partner_params=partner_params)
        step_fn.trace = trace
        rng_key, sub_key = brandom.split(rng)
        state = eval_env.init(eval_env.make_keys(sub_key, num_eval_envs))
        R = torch.zeros(num_eval_envs, dtype=torch.float32, device=eval_env.device)
        action = torch.empty(num_eval_envs, dtype=torch.int32, device=eval_env.device)
        r_actor = torch.empty_like(R)
        it = 0
        while True:
            actor = state.current_player.clone()
            logits, _ = actor_forward_pass.apply(actor_params, state.observation)
            ops.categorical(logits.contiguous(), state._mask_u8, action, None, sample=False)
            rng_key, _rng = brandom.split(rng_key)
            state = step_fn(state, action, _rng, out_state=state)
            ops.gather_reward(state.rewards, actor, r_actor, 1.0)
            R += r_actor
            it += 1
            if it % _CHECK_EVERY == 0 and bool(state._terminated_u8.all()):
                break
        if trace is not None:
            trace.append(("R", R.clone()))
        return R.mean()

    return simple_evaluate


def make_simple_duplicate_evaluate(eval_env, team1_activation, team1_model_type, team2_activation, team2_model_type,
                                   num_eval_envs, env_offset: int = 0):
    """src/evaluation.py:69-204.  `num_eval_envs` is THIS rank's shard; with
    torch.distributed initialised the statistics are all-reduced over ranks (one
    collective per match) so every rank returns the whole-match numbers."""
    team1_forward_pass = make_forward_pass(activation=team1_activation, model_type=team1_model_type)
    team2_forward_pass = make_forward_pass(activation=team2_activation, model_type=team2_model_type)

    def duplicate_evaluate(team1_params, team2_params, rng_key, trace=None, record=None, local_sums=None, team1_partner=None,
                           team2_partner=None):
        """`record` (a list) receives per step (action, table_a.terminated, table_b.terminated) BEFORE the step --
        the input of board_log.match_to_board_logs.  `local_sums` (f64[8] tensor): accumulate this rank's partial
        statistics there and skip the all-reduce (the league evaluator reduces all its matches at once).
        `team1_partner` / `team2_partner`: the net of player 1 / player 3 (of its team's architecture) instead of the team's
        net, which then plays player 0 / 2 only -- a partnership of two nets (player ids keep their team at both tables)."""
        step_fn = duplicate_step(eval_env.step)
        rng_key, sub_key = brandom.split(rng_key)
        state = _bf16_state(eval_env, eval_env.make_keys(sub_key, num_eval_envs, env_offset))  # :93-95
        table_a_info = Table_info.from_state(state)                                        # :97-112
        table_b_info = Table_info.from_state(state)
        dev = eval_env.device
        cum_return = torch.zeros(num_eval_envs, dtype=torch.float32, device=dev)
        action = torch.zeros(num_eval_envs, dtype=torch.int32, device=dev)  # finished envs keep a (no-op) Pass
        teams = _TeamRows(num_eval_envs, dev)
        while True:
            # :124-151 -- team 1's net decides for players 0/1, team 2's for players 2/3; finished envs are skipped
            rows1, rows2 = teams.split(state.current_player, state._terminated_u8)
            if rows1.shape[0] + rows2.shape[0] == 0:                                       # :120-122 ~terminated.all()
                break
            _act_team(team1_forward_pass, team1_params, team1_partner, state, action, rows1)
            _act_team(team2_forward_pass, team2_params, team2_partner, state, action, rows2)
            if trace is not None:  # tests replay the same action sequence on the oracle
                trace.append((action.clone(), None, None))
            if record is not None:
                record.append((action.cpu(), table_a_info.terminated.view(torch.uint8).cpu(),
                               table_b_info.terminated.view(torch.uint8).cpu()))
            state, table_a_info, table_b_info = step_fn(state, action, table_a_info, table_b_info)  # :164
            cum_return += state.rewards[:, 0]                                              # :167-169
        duplicate_evaluate.rows_forwarded = teams.forwarded
        if local_sums is not None:
            ops.match_stats(cum_return, local_sums)
            return None, table_a_info, table_b_info, cum_return
        sums = torch.zeros(8, dtype=torch.float64, device=dev)
        ops.match_stats(cum_return, sums)
        bdist.allreduce_sums(sums)
        mean, std_error, win_rate = bdist.stats_from_sums(sums.cpu())                      # :199-201
        log_info = (mean, std_error, win_rate)
        return log_info, table_a_info, table_b_info, cum_return

    return duplicate_evaluate


def make_league_evaluate(eval_env, activation, model_type, num_eval_envs_total: int, num_models: int):
    """The PFSP league probe of ppo.py:412-436 as ONE sharded job (BASELINE configs[4]): the learner plays a
    duplicate match against every model of the pool; the `num_eval_envs_total` envs are split into `num_models`
    equal blocks by GLOBAL env index (block m plays pool model m) and every block is sharded across the ranks, so
    the result does not depend on the rank count.  One all-reduce of f64[num_models, 8] for the whole league.
    Returns per-model (mean IMP, SE, win rate) lists -- `imp_list` / `win_rate_list` of ppo.py:414-435."""
    rank, world = bdist.rank_world()
    per_model = num_eval_envs_total // num_models
    lo, hi = bdist.shard_range(per_model, rank, world)
    matches = [make_simple_duplicate_evaluate(eval_env, activation, model_type, activation, model_type, hi - lo,
                                              env_offset=m * per_model + lo) for m in range(num_models)]

    def league_evaluate(actor_params, pool_params, rng_key):
        assert len(pool_params) == num_models
        sums = torch.zeros((num_models, 8), dtype=torch.float64, device=eval_env.device)
        for m, (match, opp) in enumerate(zip(matches, pool_params)):
            if hi > lo:
                match(actor_params, opp, rng_key, local_sums=sums[m])
        bdist.allreduce_sums(sums)
        host = sums.cpu()
        return [bdist.stats_from_sums(host[m]) for m in range(num_models)]

    return league_evaluate


# ---- self-play league over saved checkpoints (workspace/eval_selfplay_league.py) ---------------------------------------
def list_league_checkpoints(models_directory: str, exp_name: str, skip_interval: int = 100, max_step: int = 10000):
    """The script's checkpoint selection: files of `models_directory/exp_name` with "params" in the name whose step (the
    number after the first "-") is a multiple of `skip_interval` and at most `max_step`, sorted by name.  Takes ppo.train's
    `params-{i:08}.pkl` (zero-padded, so name order is step order) and leaves its `opt_state-*.pkl` out."""
    import os
    out = []
    for name in os.listdir(os.path.join(models_directory, exp_name)):
        if "params" not in name:
            continue
        try:
            step = int(name.split("-")[1].split(".")[0])
        except (IndexError, ValueError):
            raise ValueError(f"checkpoint {name!r} has no step number after its first '-'") from None
        if step % skip_interval == 0 and step <= max_step:
            out.append(name)
    return sorted(out)


def league_matrices(num_models: int, pair_imps):
    """The script's matrices from {(i, j): imp} over pairs i < j: win_lose[i, j] = -imp, win_lose[j, i] = imp; `dis` holds
    the sign (0 for a tie) and `clip` the value clipped to [-1, 1], with the same antisymmetry."""
    import numpy as np
    win_lose = np.zeros((num_models, num_models))
    win_lose_dis = np.zeros((num_models, num_models))
    win_lose_clip = np.zeros((num_models, num_models))
    for (i, j), imp in pair_imps.items():
        win_lose[i][j], win_lose[j][i] = -imp, imp
        clip_imp = np.clip(imp, -1, 1)
        win_lose_clip[i][j], win_lose_clip[j][i] = -clip_imp, clip_imp
        if imp > 0:
            win_lose_dis[i][j], win_lose_dis[j][i] = -1, 1
        elif imp < 0:
            win_lose_dis[i][j], win_lose_dis[j][i] = 1, -1
    return win_lose, win_lose_dis, win_lose_clip


# ---- the device-loop evaluators: one brl_duplicate_match call per match / league chunk (eval.py:53) -------------------------
class _MatchBuffers:
    """Fixed-address inputs and outputs of brl_duplicate_match for one shape (n envs, M nets, P ranges; P = 0: one range
    over the batch), so that repeated calls relaunch the op's cached graph instead of capturing a new one."""

    def __init__(self, n: int, M: int, P: int, dev, with_models: bool, with_tables: bool, pool=None, players: bool = False):
        self.keys = torch.empty(n, dtype=torch.int64, device=dev)
        self.pool = pool if pool is not None else torch.zeros((M, ops.mlp_pool_stride()), dtype=torch.uint8, device=dev)
        # a net per team, or with `players` per player id (BRL_F_PLAYER_MODELS)
        self.env_models = torch.empty((n, 4 if players else 2), dtype=torch.int32, device=dev) if with_models else None
        self.offsets = torch.empty(P + 1, dtype=torch.int64, device=dev) if P else None
        self.scratch = torch.empty(ops.duplicate_match_scratch_bytes(n, M), dtype=torch.uint8, device=dev)
        self.cum_return = torch.empty(n, dtype=torch.float32, device=dev)
        self.sums = torch.zeros((P, 8) if P else (8,), dtype=torch.float64, device=dev)
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)
        self.tables = (ops.TableInfoBuffers(n, dev), ops.TableInfoBuffers(n, dev)) if with_tables else (None, None)

    def prefix(self, n: int, P: int) -> "_MatchBuffers":
        """the first n envs and P ranges of these buffers (with env models and ranges, without Table_infos): a smaller shape at
        the same addresses, whose scratch is large enough because the op's scratch size grows with n"""
        v = _MatchBuffers.__new__(_MatchBuffers)
        v.keys, v.env_models, v.cum_return = self.keys[:n], self.env_models[:n], self.cum_return[:n]
        v.offsets, v.sums = self.offsets[:P + 1], self.sums[:P]
        v.pool, v.scratch, v.status, v.tables = self.pool, self.scratch, self.status, self.tables
        return v

    def play(self, eval_env, single_bf16: bool, tune: int, system_hist=None):
        self.sums.zero_()
        ops.duplicate_match(self.keys, eval_env.table, self.pool, self.scratch, self.cum_return, self.sums, self.status,
                            env_models=self.env_models, range_offsets=self.offsets, table_a=self.tables[0],
                            table_b=self.tables[1], single_bf16=single_bf16, tune=tune,
                            illegal_penalty=eval_env.illegal_penalty, illegal_bonus=eval_env.illegal_bonus,
                            system_hist=system_hist)


def _check_match_status(status: int, op: str = "brl_duplicate_match") -> None:
    if status == ops._lib.MATCH_BAD_MODEL:
        raise ops._lib.BrlError(f"{op}: an acting net id is outside [0, M)")
    if status != ops._lib.MATCH_OK:
        raise ops._lib.BrlError(f"{op}: envs still live after {ops._lib.MATCH_MAX_STEPS} steps (status {status})")


def _table_infos(tables):
    """copies of a buffer set's two final TableInfoBuffers as Table_info"""
    return [Table_info(t.terminated.clone(), t.rewards.clone(), t.last_bid.clone(), t.last_bidder.clone(), t.call_x.clone(),
                       t.call_xx.clone()) for t in tables]


def _fill_chunk(b, board_keys, g, n: int, nets) -> None:
    """keys and env_models of a chunk of global envs g: env g plays board g % n with the nets of match g // n"""
    b.keys.copy_(board_keys[torch.as_tensor(g % n, device=b.keys.device)])
    b.env_models.copy_(torch.as_tensor(nets[g // n], device=b.keys.device))


def _play_single(eval_env, sets, new_set, partnered: bool, rng_key, env_offset: int, nets, play, op: str):
    """One call of a single-match device evaluator: the buffer set of `sets` for the partner flag (allocated by
    `new_set(partnered)` at its first use), the keys of the match (src/evaluation.py:93-94), nets = [(forward_pass, params)]
    packed into pool slots 0 / 1 / 2 (None params: the slot is not read), `play(b)`, then one host copy of the all-reduced
    sums (a copy: the buffers keep theirs) with the status, or of the status alone where the set has no sums; the status is
    checked.  Returns (b, host sums or None)."""
    if partnered not in sets:
        sets[partnered] = new_set(partnered)
    b = sets[partnered]
    _, sub_key = brandom.split(rng_key)
    b.keys.copy_(eval_env.make_keys(sub_key, b.keys.shape[0], env_offset))
    blob_bytes = ops._lib.load().brl_mlp_packed_bytes()
    for slot, (forward_pass, params) in enumerate(nets):
        if params is not None:
            forward_pass.pack_into(params, b.pool[slot, :blob_bytes])
    play(b)
    if b.sums is None:
        _check_match_status(int(b.status[0]), op)
        return b, None
    sums = b.sums.clone()
    bdist.allreduce_sums(sums)
    host = torch.cat((sums, b.status.to(torch.float64))).cpu()
    _check_match_status(int(host[-1]), op)
    return b, host[:-1]


def make_device_duplicate_evaluate(eval_env, activation, model_type, num_eval_envs, env_offset: int = 0, *, tune: int = 0):
    """make_simple_duplicate_evaluate (src/evaluation.py:69-204) with the whole match in one brl_duplicate_match call: the
    loop runs on the device (a CUDA graph WHILE node), so a match costs one launch and one host read of its statistics.
    Same contract -- `duplicate_evaluate(team1_params, team2_params, rng_key) -> (log_info, table_a_info, table_b_info,
    cum_return)`, same key split and keys, one all-reduce of f64[8] over the ranks -- and the same per-env results.
    Both teams share `activation` / `model_type` (the pool holds one architecture).  `record` / `trace` need per-step host
    copies: use make_simple_duplicate_evaluate for them.  `tune`: BRL_F_TUNE_MLP_* bits pinning the forward's path.
    `team1_partner`: player 1's net instead of team1_params, which then plays player 0 only (a 3-net pool with nets by
    player id, BRL_F_PLAYER_MODELS; its own buffers and graph)."""
    forward_pass = make_forward_pass(activation=activation, model_type=model_type)
    n, dev = num_eval_envs, eval_env.device
    single_bf16 = forward_pass.precision == "tc-bf16"

    def new_set(partnered):
        if not partnered:
            return _MatchBuffers(n, 2, 0, dev, with_models=False, with_tables=True)
        b = _MatchBuffers(n, 3, 0, dev, with_models=True, with_tables=True, players=True)
        b.env_models.copy_(torch.tensor([0, 2, 1, 1], dtype=torch.int32, device=dev).expand(n, 4))
        return b

    sets = {False: new_set(False)}                              # with a partner: a 3-net set, allocated at its first call

    def duplicate_evaluate(team1_params, team2_params, rng_key, team1_partner=None):
        b, sums = _play_single(eval_env, sets, new_set, team1_partner is not None, rng_key, env_offset,
                               [(forward_pass, team1_params), (forward_pass, team2_params), (forward_pass, team1_partner)],
                               lambda b: b.play(eval_env, single_bf16, tune), "brl_duplicate_match")     # :93-198
        infos = _table_infos(b.tables)
        return bdist.stats_from_sums(sums), infos[0], infos[1], b.cum_return.clone()    # :199-201

    return duplicate_evaluate


def pair_chunk_layout(num_pairs: int, n: int, pairs_per_chunk: int, rank: int, world: int):
    """How the device pair matches lay out `num_pairs` matches of `n` boards each: chunks of `pairs_per_chunk` matches, each
    chunk's P * n envs sharded over the ranks by global env index g (match g // n, board g % n).  Yields per chunk
    (c0, P, lo, hi, p_lo, p_hi, bounds): the chunk's first pair, its pair count, this rank's global env range [lo, hi), the
    matches [p_lo, p_hi) of the chunk that range touches and their local env ranges bounds[p - p_lo] .. bounds[p - p_lo + 1]."""
    import numpy as np
    for c0 in range(0, num_pairs, pairs_per_chunk):
        P = min(pairs_per_chunk, num_pairs - c0)
        lo, hi = bdist.shard_range(P * n, rank, world)
        p_lo, p_hi = lo // n, (hi + n - 1) // n
        bounds = np.clip(np.arange(p_lo, p_hi + 1, dtype=np.int64) * n - lo, 0, hi - lo)
        yield c0, P, lo, hi, p_lo, p_hi, bounds


def _pool_match_shape(max_pairs: int, n: int, pairs_per_chunk: int, world: int):
    """(envs, ranges) of the largest chunk shard any rank plays for at most `max_pairs` matches of `n` boards"""
    P = min(max_pairs, pairs_per_chunk)
    return -(-P * n // world), P


def pair_match_bytes(n_envs: int, M: int, P: int) -> int:
    """device bytes of one set of the pair matches' buffers for n_envs envs, M nets and P ranges (the pool not counted)"""
    return ops.duplicate_match_scratch_bytes(n_envs, M) + n_envs * (8 + 8 + 4) + 8 * (P + 1) + 64 * P + 4


def pfsp_probe_bytes(capacity: int, num_eval_envs: int, max_envs: int = 1 << 20, world: int = 1) -> int:
    """device bytes make_device_pfsp_probe holds on each of `world` ranks for a zoo of `capacity` models (its pool not
    counted): one buffer set for the largest chunk over M = 1 + capacity nets"""
    if capacity == 0:
        return 0
    n_envs, P = _pool_match_shape(capacity, num_eval_envs, max(1, (max_envs * world) // num_eval_envs), world)
    return pair_match_bytes(n_envs, 1 + capacity, P)


def _make_device_pair_matches(eval_env, forward_pass, num_eval_envs: int, max_envs: int, tune: int):
    """The engine of the self-play league, the PFSP probe and cross-play: `matches(pairs, rng_key, params_list=None, pool=None,
    cum_returns=None)` plays every (i, j) of `pairs` -- net i of the pool on players 0/1, net j on 2/3 -- as the duplicate match
    `make_simple_duplicate_evaluate(..., num_eval_envs)(net_i, net_j, rng_key)` plays, on the same boards in every match, and
    returns their (imp, se, win_rate) in `pairs` order.  `pairs` may instead hold 4-tuples (a, b, c, d): net a on player 0,
    b on 1, c on 2 and d on 3 (env_models[n, 4] by player id, BRL_F_PLAYER_MODELS; with `params_list` only).  The nets are `params_list` (packed into a pool of the matches' own)
    or the caller's packed `pool` (u8[M, brl_mlp_pool_stride()], used in place).  At most `max_envs` envs per rank make one
    chunk and one brl_duplicate_match call; a chunk's envs are sharded by global index over the ranks (pair_chunk_layout),
    with one all-reduce of f64[P, 8] and one host read per chunk, so the result does not depend on the rank count.
    Buffers stay at fixed addresses, so repeated calls relaunch the op's cached graphs: with `params_list` one set per shape;
    with a caller's pool ONE set, allocated by `matches.reserve(pool, max_pairs)` for the largest chunk of up to `max_pairs`
    matches (pair_match_bytes of _pool_match_shape), every chunk playing on a prefix of it -- so a pool whose pair count grows
    call by call (a filling zoo) holds exactly that memory from the reservation on.  `cum_returns` (a dict, tests) receives
    each pair's per-env returns of this rank's shard.  `system_hist` (int64 [M, 75, 38, 96] on the device): every decision of
    this rank's shard is added to the histogram of the net that made it (brl_duplicate_match [21], one u32 histogram per chunk
    added in); the caller all-reduces it."""
    import numpy as np
    rank, world = bdist.rank_world()
    n, dev = num_eval_envs, eval_env.device
    pairs_per_chunk = max(1, (max_envs * world) // n)
    buffers = {}
    held = {}                                                   # the caller pool's set: pool, max_pairs, buffers
    blob_bytes = ops._lib.load().brl_mlp_packed_bytes()
    single_bf16 = forward_pass.precision == "tc-bf16"
    chunk_hists = {}                                            # M -> the u32 histogram one chunk counts into

    def reserve(pool, max_pairs: int) -> None:
        if held and held["pool"] is pool and held["max_pairs"] >= max_pairs:
            return
        held.clear()                                            # free the previous set before allocating the new one
        n_envs, P = _pool_match_shape(max_pairs, n, pairs_per_chunk, world)
        held.update(pool=pool, max_pairs=max_pairs,
                    buffers=_MatchBuffers(n_envs, pool.shape[0], P, dev, with_models=True, with_tables=False, pool=pool))

    def matches(pairs, rng_key, params_list=None, pool=None, cum_returns=None, system_hist=None):
        M = len(params_list) if pool is None else pool.shape[0]
        width = len(pairs[0]) if len(pairs) else 2             # nets by team (i, j) or by player (a, b, c, d)
        if width not in (2, 4) or any(len(p) != width for p in pairs) or (width == 4 and pool is not None):
            raise ValueError("matches: pairs are all (i, j), or all (a, b, c, d) with params_list")
        if pool is not None:
            reserve(pool, len(pairs))
        _, sub_key = brandom.split(rng_key)                                                # as duplicate_evaluate
        board_keys = eval_env.make_keys(sub_key, n)
        pair_arr = np.asarray(pairs, dtype=np.int32).reshape(-1, width)
        stats = []
        for c0, P, lo, hi, p_lo, p_hi, bounds in pair_chunk_layout(len(pairs), n, pairs_per_chunk, rank, world):
            sums = torch.zeros((P, 8), dtype=torch.float64, device=dev)
            status = 0
            if hi > lo:
                g = np.arange(lo, hi)
                if pool is not None:
                    b = held["buffers"].prefix(hi - lo, p_hi - p_lo)
                else:
                    key = (hi - lo, M, p_hi - p_lo, width)
                    if key not in buffers:
                        buffers[key] = _MatchBuffers(hi - lo, M, p_hi - p_lo, dev, with_models=True, with_tables=False,
                                                     players=width == 4)
                    b = buffers[key]
                    for m, params in enumerate(params_list):
                        forward_pass.pack_into(params, b.pool[m, :blob_bytes])
                _fill_chunk(b, board_keys, g, n, pair_arr[c0:])
                b.offsets.copy_(torch.as_tensor(bounds, device=dev))
                if system_hist is None:
                    b.play(eval_env, single_bf16, tune)
                else:
                    if M not in chunk_hists:
                        chunk_hists[M] = ops.new_system_hist(M, dev)
                    chunk_hist = chunk_hists[M]
                    chunk_hist.zero_()
                    b.play(eval_env, single_bf16, tune, chunk_hist)
                    system_hist += ops.system_hist_counts(chunk_hist)
                sums[p_lo:p_hi] = b.sums
                status = b.status
                if cum_returns is not None:
                    for p in range(p_lo, p_hi):
                        cum_returns[pairs[c0 + p]] = b.cum_return[int(bounds[p - p_lo]):int(bounds[p - p_lo + 1])].clone()
            bdist.allreduce_sums(sums)
            host = sums.cpu()
            _check_match_status(int(status))
            stats.extend(bdist.stats_from_sums(host[p]) for p in range(P))
        return stats

    matches.reserve = reserve
    matches.held = held
    return matches


def make_selfplay_league_evaluate(eval_env, activation, model_type, num_eval_envs: int, max_envs: int = 1 << 20, *,
                                  tune: int = 0):
    """workspace/eval_selfplay_league.py's league as batched jobs: every pair (i, j), i < j, in itertools.combinations
    order plays the match `make_simple_duplicate_evaluate(..., num_eval_envs)(params_list[i], params_list[j], rng_key)`
    plays (team 1 = i on players 0/1, team 2 = j; env e of every match keyed as local index e).  The matches of a chunk
    (at most `max_envs` envs per rank) run as ONE env batch in one brl_duplicate_match call over a pool of all the nets: the
    loop runs on the device, grouping the live rows by acting net each step for the grouped forward.  The chunk's envs are
    sharded by global index over the ranks, with one all-reduce of f64[P, 8] per chunk, so the result does not depend on the
    rank count.  `league(params_list, rng_key)` returns ({(i, j): (imp, se, win_rate)}, win_lose, win_lose_dis,
    win_lose_clip); `cum_returns` (a dict, tests) receives each pair's per-env returns of this rank's shard.  `tune`:
    BRL_F_TUNE_MLP_* bits pinning the forward's path."""
    import itertools
    matches = _make_device_pair_matches(eval_env, make_forward_pass(activation=activation, model_type=model_type),
                                        num_eval_envs, max_envs, tune)

    def league(params_list, rng_key, cum_returns=None):
        M = len(params_list)
        pairs = list(itertools.combinations(range(M), 2))
        stats = dict(zip(pairs, matches(pairs, rng_key, params_list=params_list, cum_returns=cum_returns)))
        return (stats,) + league_matrices(M, {pair: s[0] for pair, s in stats.items()})

    return league


def make_crossplay_evaluate(eval_env, activation, model_type, num_eval_envs: int, max_envs: int = 1 << 20, *, tune: int = 0):
    """Cross-play: how well the nets of a pool bid together as partners.  `crossplay(params_list, opponents, rng_key,
    cum_returns=None)` plays every ordered partnership (a, b) of the M nets of `params_list` -- net a on player 0, net b on
    player 1, the diagonal (a, a) included -- against the fixed pair `opponents` = (c, d) on players 2 / 3, each the duplicate
    match `make_simple_duplicate_evaluate(..., num_eval_envs)(a, c, rng_key, team1_partner=b, team2_partner=d)` plays, on the
    same boards in every match.  The M^2 matches are chunked and sharded as the self-play league's (at most `max_envs` envs
    per rank a chunk, one brl_duplicate_match call each over a pool of the M + 2 nets with the nets by player id), so the
    result does not depend on the rank count.  Returns ({(a, b): (imp, se, win_rate)}, imp[M, M]) with imp[a, b] the mean
    IMP of partnership (a, b); (a, a) against (c, c) is `make_device_duplicate_evaluate(...)(a, c, rng_key)`'s.
    `cum_returns` (a dict, tests) receives each partnership's per-env returns of this rank's shard under (a, b).  `tune`:
    BRL_F_TUNE_MLP_* bits pinning the forward's path."""
    import numpy as np
    matches = _make_device_pair_matches(eval_env, make_forward_pass(activation=activation, model_type=model_type),
                                        num_eval_envs, max_envs, tune)

    def crossplay(params_list, opponents, rng_key, cum_returns=None):
        M = len(params_list)
        c, d = opponents
        pairs = [(a, b, M, M + 1) for a in range(M) for b in range(M)]
        by_pair = {} if cum_returns is not None else None
        stats = dict(zip(((a, b) for a, b, _, _ in pairs),
                         matches(pairs, rng_key, params_list=list(params_list) + [c, d], cum_returns=by_pair)))
        if cum_returns is not None:
            cum_returns.update({pair[:2]: v for pair, v in by_pair.items()})
        imp = np.array([[stats[(a, b)][0] for b in range(M)] for a in range(M)], dtype=np.float64).reshape(M, M)
        return stats, imp

    return crossplay


def make_bidding_system_evaluate(eval_env, activation, model_type, num_eval_envs: int, max_envs: int = 1 << 20, *,
                                 tune: int = 0):
    """The bidding systems of M nets (DESIGN.md f15): `system(params_list, rng_key, opponent=None)` returns int64
    hist[M, 75, 38, 96] on the host, every decision of the nets' duplicate matches counted for the net that made it.  By
    default net m plays all four seats in block m (its system as it plays with and against itself); with `opponent=k` net m
    plays players 0/1 against net k on 2/3 (match m is `make_simple_duplicate_evaluate(...)(params_list[m],
    params_list[k], rng_key)`), and net k's decisions in every match count for net k.  Every match is played on the same
    boards.  The matches run on the pair-match engine (at most `max_envs` envs per rank a chunk, one brl_duplicate_match
    call each, sharded by global env index) with one int64 all-reduce of the histogram per call, so the result does not
    depend on the rank count.  `tune`: BRL_F_TUNE_MLP_* bits pinning the forward's path."""
    matches = _make_device_pair_matches(eval_env, make_forward_pass(activation=activation, model_type=model_type),
                                        num_eval_envs, max_envs, tune)

    def system(params_list, rng_key, opponent=None):
        M = len(params_list)
        if opponent is not None and not 0 <= opponent < M:
            raise ValueError(f"make_bidding_system_evaluate: opponent {opponent} is not a net of the {M} given")
        pairs = [(m, m if opponent is None else opponent) for m in range(M)]
        hist = torch.zeros((M,) + ops.SYSTEM_SHAPE, dtype=torch.int64, device=eval_env.device)
        matches(pairs, rng_key, params_list=params_list, system_hist=hist)
        bdist.allreduce_sums(hist)
        return hist.cpu().numpy()

    return system


def call_values_bytes(n_envs: int, M: int, record_capacity: int = 0) -> int:
    """device bytes of one chunk of make_call_values_evaluate for n_envs base envs and M nets (its pool not counted): the keys,
    env_models, the two matches' scratch, cum_return, sums, status, both Table_infos, the int64 sums and the records"""
    table_info = n_envs * (1 + 16 + 4 + 4 + 1 + 1)
    sums = 8 * M * (ops._lib.SYS_CONTEXTS * (38 * 38 * 4 + 4) + 1)
    records = record_capacity * (6 * 4 + 38 * 4) + 8 if record_capacity else 0
    return (n_envs * (8 + 8 + 4) + ops.duplicate_match_scratch_bytes(n_envs, M) + 64 + 4 + 2 * table_info
            + ops.call_values_scratch_bytes(n_envs, M) + sums + 4 + records)


class _CallValueBuffers:
    """Fixed-address buffers of one chunk shape (n base envs, M nets): the base match (brl_duplicate_match with its Table_infos)
    and brl_call_values, so repeated calls relaunch both ops' cached graphs."""

    def __init__(self, n: int, M: int, dev):
        self.match = _MatchBuffers(n, M, 0, dev, with_models=True, with_tables=True)
        self.scratch = torch.empty(ops.call_values_scratch_bytes(n, M), dtype=torch.uint8, device=dev)
        self.gain = torch.empty((M,) + ops.CALL_GAIN_SHAPE, dtype=torch.int64, device=dev)
        self.regret = torch.empty((M,) + ops.CALL_REGRET_SHAPE, dtype=torch.int64, device=dev)
        self.mismatch = torch.empty(M, dtype=torch.int64, device=dev)
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)
        self.records = None


def make_call_values_evaluate(eval_env, activation, model_type, num_eval_envs: int, max_envs: int = 1 << 20, *, tune: int = 0):
    """Counterfactual call values of M nets (DESIGN.md f16): `call_values(params_list, rng_key, opponent=None, records=False)`
    plays the matches make_bidding_system_evaluate plays (net m in all four seats, or net m on players 0/1 against net k =
    `opponent` on 2/3, every match on the same boards) and at every decision plays out every legal alternative call.  Returns
    a dict of host int64 arrays: `gain_sums` [M, 75, 38, 38, 4] = {n, sum g, sum g^2, #(g > 0)} per (net, context, played,
    alternative), `regret_sums` [M, 75, 4] = {decisions, sum regret, sum regret^2, #(regret > 0)} and `mismatch` [M]; with
    `records=True` also this rank's decision records (dict of arrays env, table, player, net, context, played, r[., 38]; env =
    global base env index m * num_eval_envs + board).  `records="train"` also returns this rank's training examples
    (DESIGN.md f17) as device tensors, `examples` = dict(obs bf16 [k, 480], gain f32 [k, 38] (NaN: illegal), net int32 [k]),
    row k belonging to record k; the records and examples are then ordered by env, table and play order, so that a seeded
    run repeats them row for row.  `matches`: the (net on players 0/1, net on players 2/3) pairs to play instead, match j on
    global base envs j * num_eval_envs + board (e.g. [(0, 1)]: only net 0 against net 1).
    The M * num_eval_envs base envs are sharded over the ranks by global index (as the pair-match engine does), and each
    rank plays its share in chunks of at most max_envs // 38 base envs, so that a chunk's 38 branch slots per env fit
    `max_envs` branch rows.  Per chunk: one brl_duplicate_match (the base results) and one brl_call_values call; a chunk
    holds call_values_bytes(chunk, M) device bytes.  The int64 sums are integers added in any order, with one all-reduce per
    call, so they do not depend on the chunking or the rank count.  `tune`: BRL_F_TUNE_MLP_* bits pinning the forward."""
    import numpy as np
    forward_pass = make_forward_pass(activation=activation, model_type=model_type)
    n, dev = num_eval_envs, eval_env.device
    chunk = max(1, max_envs // ops.NUM_ACTIONS)
    single_bf16 = forward_pass.precision == "tc-bf16"
    blob_bytes = ops._lib.load().brl_mlp_packed_bytes()
    buffers = {}

    def call_values(params_list, rng_key, opponent=None, records=False, matches=None):
        M = len(params_list)
        if M < 1:
            raise ValueError("make_call_values_evaluate: no nets given")
        if opponent is not None and not 0 <= opponent < M:
            raise ValueError(f"make_call_values_evaluate: opponent {opponent} is not a net of the {M} given")
        if matches is not None and (opponent is not None or not matches or
                                    any(len(mt) != 2 or not all(0 <= x < M for x in mt) for mt in matches)):
            raise ValueError(f"make_call_values_evaluate: matches must be (net on players 0/1, net on 2/3) pairs of the {M} "
                             "nets, without `opponent`")
        if records not in (False, True, "train"):
            raise ValueError(f"make_call_values_evaluate: records must be False, True or 'train', got {records!r}")
        rank, world = bdist.rank_world()
        _, sub_key = brandom.split(rng_key)                                                # as duplicate_evaluate
        board_keys = eval_env.make_keys(sub_key, n)
        train = records == "train"
        examples = []
        pairs = np.array(matches if matches is not None else [(m, m if opponent is None else opponent) for m in range(M)],
                         dtype=np.int32).reshape(-1, 2)
        total = torch.zeros(M * (int(np.prod(ops.CALL_GAIN_SHAPE)) + int(np.prod(ops.CALL_REGRET_SHAPE)) + 1), dtype=torch.int64,
                            device=dev)
        n_gain, n_regret = M * int(np.prod(ops.CALL_GAIN_SHAPE)), M * int(np.prod(ops.CALL_REGRET_SHAPE))
        recs = []
        lo, hi = bdist.shard_range(len(pairs) * n, rank, world)
        for c0 in range(lo, hi, chunk):
            c1 = min(hi, c0 + chunk)
            key = (c1 - c0, M)
            if key not in buffers:
                buffers[key] = _CallValueBuffers(c1 - c0, M, dev)
            b = buffers[key]
            for m, params in enumerate(params_list):
                forward_pass.pack_into(params, b.match.pool[m, :blob_bytes])
            g = np.arange(c0, c1)
            _fill_chunk(b.match, board_keys, g, n, pairs)
            b.match.play(eval_env, single_bf16, tune)
            if records and (b.records is None or b.records.train != train):
                b.records = ops.CallValueRecords(48 * (c1 - c0), dev, train)  # about twice a typical board's decisions
            while True:
                ops.call_values(b.match.keys, eval_env.table, b.match.pool, b.match.env_models, b.match.tables[0].rewards,
                                b.match.tables[1].rewards, b.scratch, b.gain, b.regret, b.mismatch, b.status,
                                records=b.records if records else None, env_offset=c0, single_bf16=single_bf16, tune=tune,
                                illegal_penalty=eval_env.illegal_penalty, illegal_bonus=eval_env.illegal_bonus)
                status = int(torch.maximum(b.status, b.match.status)[0])
                if status != ops._lib.MATCH_RECORD_CAPACITY:
                    break
                b.records = ops.CallValueRecords(int(b.records.count[0]), dev, train)  # grow to the chunk's decisions
            _check_match_status(status, "brl_call_values")
            total[:n_gain] += b.gain.view(-1)
            total[n_gain:n_gain + n_regret] += b.regret.view(-1)
            total[n_gain + n_regret:] += b.mismatch
            if records:
                k = int(b.records.count[0])
                if not train:
                    recs.append({f: getattr(b.records, f)[:k].cpu().numpy() for f in ops.CALL_RECORD_FIELDS + ("r",)})
                else:
                    # the slots follow the gains kernel's atomics; an (env, table)'s slots rise in play order, so a stable
                    # sort by (env, table) gives an order that a seeded run repeats.  Gathered copies: the buffers are
                    # reused by the next chunk and the next call.
                    r = b.records
                    order = torch.sort(r.env[:k].long() * 2 + r.table[:k], stable=True).indices
                    recs.append({f: getattr(r, f)[:k][order].cpu().numpy() for f in ops.CALL_RECORD_FIELDS + ("r",)})
                    examples.append((r.obs[:k][order], r.gain[:k][order], r.net[:k][order]))
        bdist.allreduce_sums(total)
        host = total.cpu().numpy()
        out = dict(gain_sums=host[:n_gain].reshape((M,) + ops.CALL_GAIN_SHAPE),
                   regret_sums=host[n_gain:n_gain + n_regret].reshape((M,) + ops.CALL_REGRET_SHAPE),
                   mismatch=host[n_gain + n_regret:])
        if records:
            out["records"] = {f: np.concatenate([r[f] for r in recs]) if recs else np.zeros((0,) + ((38,) if f == "r" else ()))
                              for f in ops.CALL_RECORD_FIELDS + ("r",)}
        if train:
            out["examples"] = dict(
                obs=torch.cat([e[0] for e in examples]) if examples else torch.zeros((0, ops.OBS_DIM), dtype=torch.bfloat16, device=dev),
                gain=torch.cat([e[1] for e in examples]) if examples else torch.zeros((0, 38), dtype=torch.float32, device=dev),
                net=torch.cat([e[2] for e in examples]) if examples else torch.zeros(0, dtype=torch.int32, device=dev))
        return out

    return call_values


def make_device_pfsp_probe(eval_env, activation, model_type, num_eval_envs: int, max_envs: int = 1 << 20, *, tune: int = 0):
    """The PFSP probe of ppo.py:412-436 -- the learner against every model of a zoo.ModelZoo -- as one brl_duplicate_match
    call per chunk over the zoo's own pool (M = 1 + capacity nets, nothing copied per call).  The learner's parameters are
    re-packed into the zoo's slot 0, and block k of `num_eval_envs` envs plays (0, slot(k)) on the same boards for every k.
    `probe(current_params, zoo, rng_key) -> [(imp, se, win_rate)] * len(zoo)` in logical zoo order; entry k equals
    `make_simple_duplicate_evaluate(..., num_eval_envs)(current_params, <zoo model k>, rng_key)[0]`.  The probe holds one
    buffer set sized for the zoo's capacity (pfsp_probe_bytes), allocated by `probe.reserve(zoo)` or at the first call, so a
    filling zoo allocates nothing more.  `cum_returns` (a dict, tests) receives model k's per-env returns of this rank's
    shard under key k."""
    matches = _make_device_pair_matches(eval_env, make_forward_pass(activation=activation, model_type=model_type),
                                        num_eval_envs, max_envs, tune)

    def reserve(zoo) -> None:
        """allocate the probe's buffers for the zoo's whole capacity now (pfsp_probe_bytes); a probe call does it otherwise"""
        if zoo.capacity:
            matches.reserve(zoo.pool, zoo.capacity)

    def probe(current_params, zoo, rng_key, cum_returns=None):
        if len(zoo) == 0:
            return []
        reserve(zoo)
        zoo.set_learner(current_params)
        pairs = [(0, zoo.slot(k)) for k in range(len(zoo))]
        by_pair = {} if cum_returns is not None else None
        stats = matches(pairs, rng_key, pool=zoo.pool, cum_returns=by_pair)
        if cum_returns is not None:
            cum_returns.update({k: by_pair[pair] for k, pair in enumerate(pairs) if pair in by_pair})
        return stats

    probe.reserve = reserve
    probe.buffers = lambda: matches.held.get("buffers")      # the buffer set the probe holds (tests, memory accounting)
    return probe


# ---- full evaluation statistics (src/evaluation.py:207-1115) --------------------------------------
_S_TABLE, _S_BIDS, _S_CONTRACTS = 11, 29, 99


def _log_info_from_sums(sums, duplicate: bool):
    """The `log_info` tuple of src/evaluation.py:575-596 (evaluate) / :986-1027 (duplicate_evaluate)
    from the all-reduced partial sums of brl_eval_summary."""
    import numpy as np
    s = np.asarray(sums, dtype=np.float64)
    n = s[0]
    mean_cum = s[1] / n
    bids = s[_S_BIDS:_S_BIDS + 70] / n
    ca, cb = s[_S_CONTRACTS:_S_CONTRACTS + 70] / n, s[_S_CONTRACTS + 70:_S_CONTRACTS + 140] / n
    ta, tb = s[_S_TABLE:_S_TABLE + 9] / n, s[_S_TABLE + 9:_S_TABLE + 18] / n
    if not duplicate:
        return (mean_cum, s[4] / n, s[5] / n, s[6] / n, bids[:35], bids[35:], ca[:35], ca[35:],
                ca[:35].sum(), ca[35:].sum(), ta[1], ta[2], ta[3], ta[4], ta[5], ta[6], ta[7], ta[8], ta[0])
    var = max(0.0, (s[2] - s[1] * s[1] / n) / (n - 1)) if n > 1 else float("nan")
    std_error = np.sqrt(var) / np.sqrt(n)
    half = lambda x, y: (x + y) / 2  # noqa: E731
    return (mean_cum, std_error, half(s[9] / n, s[10] / n), s[4] / n, s[5] / n, s[6] / n, bids[:35] / 2, bids[35:] / 2,
            half(ca[:35], cb[:35]), half(ca[35:], cb[35:]), half(ca[:35].sum(), cb[:35].sum()),
            half(ca[35:].sum(), cb[35:].sum()), half(ta[1], tb[1]), half(ta[2], tb[2]), half(ta[3], tb[3]),
            half(ta[4], tb[4]), half(ta[5], tb[5]), half(ta[6], tb[6]), half(ta[7], tb[7]), half(ta[8], tb[8]),
            half(ta[0], tb[0]), s[7] / n, s[8] / n)


def make_evaluate(eval_env, team1_activation, team1_model_type, team2_activation, team2_model_type, team2_model_path,
                  num_eval_envs, game_mode, duplicate=False, team2_params=None, env_offset: int = 0):
    """src/evaluation.py:207-1032.  Team 1 (`actor_params`, players 0/1) against a fixed team 2 (the pickle at
    `team2_model_path`, or always-pass in "free-run"); every decision is the masked argmax.  Besides the score it
    logs, per team, the unmasked probability mass on illegal actions, bid / contract histograms and declarer /
    double / make / down / pass-out ratios.  `num_eval_envs` is this rank's shard; the statistics are all-reduced
    (one collective) when torch.distributed is initialised.  Both evaluators take `partner_params`: player 1's net (of the
    actor's architecture) instead of the actor, which then plays player 0 only."""
    actor_forward_pass = make_forward_pass(activation=team1_activation, model_type=team1_model_type)
    opp_forward_pass = make_forward_pass(activation=team2_activation, model_type=team2_model_type)
    opp_params = _opponent_params(eval_env, team2_params, team2_model_path, game_mode)
    n, dev = num_eval_envs, eval_env.device
    n_sums = ops._lib.load().brl_eval_num_sums()

    def _loop(actor_params, rng_key, step, state, trace, partner_params):
        acc = torch.zeros((n, ops._lib.EVAL_ACC_COLS), dtype=torch.float32, device=dev)
        cum_return = torch.zeros(n, dtype=torch.float32, device=dev)
        rewards = torch.zeros((n, 4), dtype=torch.float32, device=dev)
        action = torch.zeros(n, dtype=torch.int32, device=dev)
        # each live env's row holds the logits of the team that acts there (scattered by the listed forward)
        logits = torch.zeros((n, ops.NUM_ACTIONS), dtype=torch.float32, device=dev)
        teams = _TeamRows(n, dev)
        while True:
            rows1, rows2 = teams.split(state.current_player, state._terminated_u8)
            if rows1.shape[0] + rows2.shape[0] == 0:
                return state, acc, cum_return, rewards
            _act_team(actor_forward_pass, actor_params, partner_params, state, action, rows1, logits=logits)
            if opp_params is not None:
                opp_forward_pass.act_rows(opp_params, state.observation, state._mask_u8, action, rows2, logits=logits)
            # the step's decision + update_log_info (unmasked-softmax illegal mass, bid histograms) from the acting
            # team's logits; free-run: team 2 always passes
            ops.eval_act_log(logits, logits if opp_params is not None else None, state._mask_u8, state.current_player,
                             state._terminated_u8, action, acc, indicator_bids=not duplicate)
            if trace is not None:
                lg = logits.clone()  # row i = the logits of the team acting in env i
                trace.append((action.clone(), lg, lg if opp_params is not None else None))
            state = step(state, action)
            rewards += state.rewards
            cum_return += state.rewards[:, 0]

    def evaluate(actor_params, rng_key, trace=None, partner_params=None):
        rng_key, sub_key = brandom.split(rng_key)
        state = _bf16_state(eval_env, eval_env.make_keys(sub_key, n, env_offset))
        state, acc, cum_return, rewards = _loop(actor_params, rng_key, lambda s, a: eval_env.step(s, a, inplace=True),
                                                state, trace, partner_params)
        f = ops.state_fields(state._packed)
        sums = torch.zeros(n_sums, dtype=torch.float64, device=dev)
        ops.eval_summary(acc, cum_return, f["step_count"],
                         (f["last_bid"], f["last_bidder"], f["call_x"], f["call_xx"], None, f["pass_num"]), None, sums)
        bdist.allreduce_sums(sums)
        state.rewards.copy_(rewards)                                                   # state.replace(rewards=rewards), :574
        return state, _log_info_from_sums(sums.cpu().numpy(), duplicate=False)

    def duplicate_evaluate(actor_params, rng_key, trace=None, partner_params=None):
        step_fn = duplicate_step(eval_env.step)
        rng_key, sub_key = brandom.split(rng_key)
        state = _bf16_state(eval_env, eval_env.make_keys(sub_key, n, env_offset))
        infos = [Table_info.from_state(state), Table_info.from_state(state)]

        def step(s, a):
            s, infos[0], infos[1] = step_fn(s, a, infos[0], infos[1])
            return s

        state, acc, cum_return, _ = _loop(actor_params, rng_key, step, state, trace, partner_params)
        f = ops.state_fields(state._packed)
        sums = torch.zeros(n_sums, dtype=torch.float64, device=dev)
        tv = lambda t: (t.last_bid, t.last_bidder, t.call_x.view(torch.uint8), t.call_xx.view(torch.uint8), t.rewards, None)  # noqa: E731
        ops.eval_summary(acc, cum_return, f["step_count"], tv(infos[0]), tv(infos[1]), sums)
        bdist.allreduce_sums(sums)
        return _log_info_from_sums(sums.cpu().numpy(), duplicate=True), infos[0], infos[1]

    return duplicate_evaluate if duplicate else evaluate


_LOG_KEYS_DUP = ("eval/IMP_reward", "eval/IMP_SE", "eval/score_reward", "eval/actor_illegal_action_probs",
                 "eval/opp_illegal_action_probs", "eval/step count", None, None, None, None, "eval/actor_declarer_ratio",
                 "eval/opp_declarer_ratio", "eval/actor_doubled_ratio", "eval/actor_redoubled_ratio", "eval/opp_doubled_ratio",
                 "eval/opp_redoubled_ratio", "eval/actor_make_contract_ratio", "eval/opp_make_contract_ratio",
                 "eval/actor_down_contract_ratio", "eval/opp_down_contract_ratio", "eval/pass_out_ratio",
                 "eval/actor_pass_ratio", "eval/opp_pass_ratio")


def make_evaluate_log(log_info):
    """src/evaluation.py:1035-1115: the wandb dict of a duplicate evaluation (same keys)."""
    if len(log_info) != len(_LOG_KEYS_DUP):
        raise ValueError("make_evaluate_log expects the 23-entry log_info of duplicate_evaluate")
    log = {k: v for k, v in zip(_LOG_KEYS_DUP, log_info) if k is not None}
    actor_bid, opp_bid, actor_contract, opp_contract = log_info[6:10]
    groups = (("actor_bid_probs", actor_bid), ("actor_contract_probs", actor_contract), ("opp_bid_probs", opp_bid),
              ("opp_contract_probs", opp_contract))
    for name, vec in groups:
        index = 0
        for number in range(1, 8):
            for suit in ("C", "D", "H", "S", "NT"):
                log[f"eval/{name}/{number}{suit}"] = vec[index]
                index += 1
    return log


# ---- the device-loop twins of make_evaluate / make_simple_evaluate: one brl_evaluate_match call each (ppo.py:365-374) ----------
class _EvalBuffers:
    """Fixed-address inputs and outputs of brl_evaluate_match for one shape and mode (as _MatchBuffers: repeated calls
    relaunch the op's cached graph)."""

    def __init__(self, n: int, mode: int, dev, partner: bool = False):
        L = ops._lib
        self.mode, self.partner = mode, partner
        self.keys = torch.empty(n, dtype=torch.int64, device=dev)
        self.pool = torch.zeros((3 if partner else 2, ops.mlp_pool_stride()), dtype=torch.uint8, device=dev)
        self.scratch = torch.empty(ops.evaluate_match_scratch_bytes(n, mode, partner), dtype=torch.uint8, device=dev)
        self.cum_return = torch.empty(n, dtype=torch.float32, device=dev)
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)
        full = mode != L.EVAL_MATCH_SIMPLE
        self.acc = torch.empty((n, L.EVAL_ACC_COLS), dtype=torch.float32, device=dev) if full else None
        self.sums = torch.zeros(L.load().brl_eval_num_sums(), dtype=torch.float64, device=dev) if full else None
        dup = mode == L.EVAL_MATCH_DUPLICATE
        self.tables = (ops.TableInfoBuffers(n, dev), ops.TableInfoBuffers(n, dev)) if dup else (None, None)
        single = mode == L.EVAL_MATCH_SINGLE
        self.final_state = ops.new_state(n, dev) if single else None
        self.final = ops.EnvOutputs(n, dev, torch.bfloat16) if single else None

    def play(self, eval_env, single_bf16: bool, free_run: bool, tune: int):
        if self.sums is not None:
            self.sums.zero_()
        ops.evaluate_match(self.keys, eval_env.table, self.pool, self.scratch, self.cum_return, self.status, mode=self.mode,
                           acc=self.acc, sums=self.sums, table_a=self.tables[0], table_b=self.tables[1],
                           final_state=self.final_state, final=self.final, free_run=free_run, partner=self.partner,
                           single_bf16=single_bf16, tune=tune,
                           illegal_penalty=eval_env.illegal_penalty, illegal_bonus=eval_env.illegal_bonus)


def _one_precision(actor_forward_pass, opp_forward_pass) -> bool:
    """the single_bf16 flag of a pool holding both nets (it holds one architecture and one precision)"""
    if actor_forward_pass.precision != opp_forward_pass.precision:
        raise ValueError("the device evaluation runs both teams in one precision")
    return actor_forward_pass.precision == "tc-bf16"


def make_device_evaluate(eval_env, team1_activation, team1_model_type, team2_activation, team2_model_type, team2_model_path,
                         num_eval_envs, game_mode, duplicate=False, team2_params=None, env_offset: int = 0, *, tune: int = 0):
    """make_evaluate (src/evaluation.py:207-1032) with the whole loop in one brl_evaluate_match call: the loop runs on the
    device (a CUDA graph WHILE node), so an evaluation costs one launch and one host read of its statistics.  Same contract --
    `duplicate_evaluate(actor_params, rng_key) -> (log_info, table_a_info, table_b_info)` or `evaluate(actor_params, rng_key) ->
    (state, log_info)`, same key split and keys, `env_offset` sharding, one all-reduce of the statistics over the ranks -- and
    the same per-env results.  In "free-run" team 2's rows are forwarded by the actor's net and not read (brl_evaluate_match).
    `trace` needs per-step host copies: use make_evaluate for it.  `tune`: BRL_F_TUNE_MLP_* bits pinning the forward's path.
    `partner_params`: player 1's net instead of the actor (BRL_F_EVAL_PARTNER, its own buffers and graph).
    The returned function's `buffers` hold the last call's per-env `acc` rows and `cum_return`."""
    L = ops._lib
    actor_forward_pass = make_forward_pass(activation=team1_activation, model_type=team1_model_type)
    opp_forward_pass = make_forward_pass(activation=team2_activation, model_type=team2_model_type)
    opp_params = _opponent_params(eval_env, team2_params, team2_model_path, game_mode)
    single_bf16 = _one_precision(actor_forward_pass, opp_forward_pass)
    n, dev = num_eval_envs, eval_env.device
    mode = L.EVAL_MATCH_DUPLICATE if duplicate else L.EVAL_MATCH_SINGLE
    sets = {False: _EvalBuffers(n, mode, dev)}                  # with a partner: a 3-net set, allocated at its first call

    def play(actor_params, rng_key, partner_params):
        fn.buffers, sums = _play_single(
            eval_env, sets, lambda partnered: _EvalBuffers(n, mode, dev, partner=partnered), partner_params is not None,
            rng_key, env_offset,
            [(actor_forward_pass, actor_params), (opp_forward_pass, opp_params), (actor_forward_pass, partner_params)],
            lambda b: b.play(eval_env, single_bf16, opp_params is None, tune), "brl_evaluate_match")
        return sums.numpy()

    def evaluate(actor_params, rng_key, partner_params=None):
        sums = play(actor_params, rng_key, partner_params)
        from .env import State
        out = ops.EnvOutputs(n, dev, torch.bfloat16)
        for k in ops.EnvOutputs.__slots__:
            getattr(out, k).copy_(getattr(fn.buffers.final, k))
        return State(eval_env, fn.buffers.final_state.clone(), out), _log_info_from_sums(sums, duplicate=False)

    def duplicate_evaluate(actor_params, rng_key, partner_params=None):
        sums = play(actor_params, rng_key, partner_params)
        infos = _table_infos(fn.buffers.tables)
        return _log_info_from_sums(sums, duplicate=True), infos[0], infos[1]

    fn = duplicate_evaluate if duplicate else evaluate
    fn.buffers = sets[False]
    return fn


def par_statistics(eval_env, init_state, table_a_info, table_b_info) -> dict:
    """Bidding against the double-dummy par (DESIGN.md f13) in a duplicate match, from the match's initial state (table A's)
    and the two Table_infos a duplicate evaluator returned, for the team of player ids {0, 1} over the 2n tables:
    `imp_vs_par` (mean, standard error) of IMP(score - par) -- the other team's is its exact negative --, `abs_imp_vs_par`
    the mean |IMP vs par| and `par_contract_rate` the fraction of tables whose final contract is the par contract in level,
    strain and declaring side (doubles ignored; two passed-out boards match).  One brl_par_stats kernel forms the f64 sums and
    one all-reduce adds them over the ranks, so the result does not depend on the rank count."""
    sums = torch.zeros(8, dtype=torch.float64, device=eval_env.device)
    a, b = table_a_info, table_b_info
    ops.par_stats(init_state._packed, eval_env.table, a.rewards, a.last_bid, a.last_bidder, b.rewards, b.last_bid, b.last_bidder,
                  sums)
    bdist.allreduce_sums(sums)
    s = sums.cpu().numpy()
    mean, se, _ = bdist.stats_from_sums((s[0], s[1], s[2], 0.0))
    return {"imp_vs_par": (mean, se), "abs_imp_vs_par": s[3] / s[0], "par_contract_rate": s[4] / s[0]}


def make_device_simple_evaluate(eval_env, team1_activation, team1_model_type, team2_activation, team2_model_type,
                                team2_model_path, num_eval_envs, team2_params=None, *, tune: int = 0):
    """make_simple_evaluate (src/evaluation.py:11-66) as one brl_evaluate_match call: the same keys and per-env returns R, and
    `simple_evaluate(actor_params, rng) -> R.mean()`.  Every decision is an argmax and the net acting is fixed per seat, so the
    device loop takes one env step per iteration and forwards each live env through the one net that acts there, where the
    host loop forwards both nets over every env until the last auction ends.  `trace` needs per-step host copies: use
    make_simple_evaluate for it.  `partner_params`: the net of the initial player's partner instead of the actor
    (BRL_F_EVAL_PARTNER, its own buffers and graph).  The returned function's `buffers.cum_return` holds the last call's R."""
    L = ops._lib
    actor_forward_pass = make_forward_pass(activation=team1_activation, model_type=team1_model_type)
    opp_forward_pass = make_forward_pass(activation=team2_activation, model_type=team2_model_type)
    opp_params = _opponent_params(eval_env, team2_params, team2_model_path)
    single_bf16 = _one_precision(actor_forward_pass, opp_forward_pass)

    def new_set(partnered):
        return _EvalBuffers(num_eval_envs, L.EVAL_MATCH_SIMPLE, eval_env.device, partner=partnered)

    sets = {False: new_set(False)}

    def simple_evaluate(actor_params, rng, partner_params=None):
        simple_evaluate.buffers, _ = _play_single(
            eval_env, sets, new_set, partner_params is not None, rng, 0,
            [(actor_forward_pass, actor_params), (opp_forward_pass, opp_params), (actor_forward_pass, partner_params)],
            lambda b: b.play(eval_env, single_bf16, False, tune), "brl_evaluate_match")
        return simple_evaluate.buffers.cum_return.mean()

    simple_evaluate.buffers = sets[False]
    return simple_evaluate
