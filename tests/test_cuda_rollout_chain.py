"""GPU: back-to-back `brl_rollout_random` launches (programmatic dependent launch: each launch may start while the previous
kernel of the stream drains) compute exactly what the same calls compute one at a time, with the stream drained between
them, in all six streams, the statistics and the final state; torch kernels between and after the launches see their
inputs and outputs in stream order."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SEED = 20241017
OFFSET = 17
NAMES = ("observation", "mask", "rewards", "terminated", "current_player", "action", "stats", "state")


def _setup(n):
    from brl_b200 import ops
    from brl_b200.deals import synthetic_deal_table
    table = torch.as_tensor(synthetic_deal_table(100_000, seed=0), device=DEV)
    state, out0 = ops.new_state(n, DEV), ops.EnvOutputs(n, DEV)
    ops.init(ops.make_keys(SEED, n, DEV, env_offset=OFFSET), table, state, out0)
    torch.cuda.synchronize()
    return ops, table, state


def _run(ops, table, state, calls, sync):
    """calls: list of (k, seed, step0, uniforms or None, edit or None); edit(state, table) runs as torch kernels before the
    call.  Every call writes fresh outputs; returns each call's outputs and the state after it, all cloned in stream order."""
    n = state.shape[1]
    # allocated up front: freeing a trajectory synchronises the device, which would break the chain
    bufs = [(ops.EnvOutputs(n, DEV, rows=k), torch.empty((k, n), dtype=torch.int32, device=DEV),
             torch.zeros(4, dtype=torch.int64, device=DEV)) for k, *_ in calls]
    torch.cuda.synchronize()
    res = []
    for (k, seed, step0, uniforms, edit), (traj, act, stats) in zip(calls, bufs):
        if edit is not None:
            edit(state, table)
        ops.rollout_random(state, table, k, traj, seed=seed, step0=step0, env_offset=OFFSET, action_out=act, stats=stats,
                           uniforms=uniforms)
        # the clones are torch kernels queued right behind the launch: they must see it complete
        res.append([t.clone() for t in (traj.observation, traj.legal_action_mask, traj.rewards, traj.terminated,
                                        traj.current_player, act, stats, state)])
        if sync:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    return res


def _check(n, calls):
    ops, table, state0 = _setup(n)
    ref = _run(ops, table.clone(), state0.clone(), calls, sync=True)
    got = _run(ops, table.clone(), state0.clone(), calls, sync=False)
    for c, (r, g) in enumerate(zip(ref, got)):
        for name, a, b in zip(NAMES, r, g):
            assert torch.equal(a, b), f"call {c}: {name}"


@pytest.mark.parametrize("n", [8192, 1001])
@pytest.mark.parametrize("k", [32, 1])
def test_chained_launches_equal_serialised(n, k):
    _check(n, [(k, SEED, i * k, None, None) for i in range(8)])


def _uniforms(k, n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(-2 ** 31, 2 ** 31, (k, n), dtype=torch.int32, generator=g).to(DEV)


@pytest.mark.parametrize("n", [8192, 1001])
def test_chained_launches_with_torch_kernels_between(n):
    """state and table edited by torch between launches, steps that do not follow on, a new seed, k changing, caller-supplied
    uniforms mixed with Philox launches"""
    def edit_state(state, table):  # one env's state words: a restart of env 5 from env 3's state
        state[:, 5] = state[:, 3]

    def edit_table(state, table):  # deal rows edited in place: every env's deal index now names another deal
        table.copy_(torch.roll(table, 1, dims=0))

    def foreign(state, table):  # an unrelated torch kernel on the stream
        torch.empty(1 << 20, device=DEV).fill_(1.0)

    u8, u5 = _uniforms(8, n, 1), _uniforms(5, n, 2)
    calls = [(32, SEED, 0, None, None), (32, SEED, 32, None, edit_state), (32, SEED, 96, None, None),
             (32, SEED + 1, 128, None, None), (8, SEED + 1, 160, None, edit_table), (8, SEED + 1, 168, u8, None),
             (5, SEED + 1, 176, u5, foreign), (32, SEED + 1, 181, None, foreign), (1, SEED + 1, 213, None, None),
             (40, SEED + 1, 214, None, edit_state)]
    _check(n, calls)


def test_chain_matches_oracle():
    """the chained launches against the C oracle's rollout, call by call"""
    import numpy as np
    from oracle import oracle as orc
    from brl_b200 import ops
    from brl_b200.deals import synthetic_deal_table
    n, k, seed, offset = 1001, 7, 4242, 1000
    table = synthetic_deal_table(2000, seed=11)
    env = orc.OracleEnv(table, n)
    env.init(orc.make_keys(seed, n, offset))
    table_t = torch.as_tensor(table, device=DEV)
    state, out0 = ops.new_state(n, DEV), ops.EnvOutputs(n, DEV)
    ops.init(ops.make_keys(seed, n, DEV, env_offset=offset), table_t, state, out0)
    outs = [(ops.EnvOutputs(n, DEV, rows=k), torch.empty((k, n), dtype=torch.int32, device=DEV)) for _ in range(6)]
    torch.cuda.synchronize()
    for c, (traj, act) in enumerate(outs):
        ops.rollout_random(state, table_t, k, traj, seed=seed, step0=c * k, env_offset=offset, action_out=act)
    torch.cuda.synchronize()
    for c, (traj, act) in enumerate(outs):
        ref = env.rollout_random(seed, c * k, k, env_offset=offset)
        assert (act.cpu().numpy() == ref["action"]).all(), c
        assert (traj.observation.cpu().numpy() == ref["observation"]).all(), c
        assert (traj.legal_action_mask.cpu().numpy() == ref["legal_action_mask"]).all(), c
        assert (traj.rewards.cpu().numpy() == ref["rewards"]).all(), c
        assert (traj.terminated.cpu().numpy() == ref["terminated"]).all(), c
    p = env.export_private()
    f = ops.state_fields(state)
    for name in ("deal", "dealer", "last_bid", "pass_num", "step_count"):
        assert (f[name].cpu().numpy() == np.asarray(p[name])).all(), name
