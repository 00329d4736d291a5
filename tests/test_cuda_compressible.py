"""GPU: rollout trajectories in compressible device memory (brl_alloc_compressible) receive exactly what plain torch
allocations receive, and the allocator gives its memory back."""
import gc

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SEED = 20241017


def _rollout(ops, table, state0, traj, k, uniforms):
    state = state0.clone()
    n = state.shape[1]
    act = torch.empty((k, n), dtype=torch.int32, device=DEV)
    stats = torch.zeros(4, dtype=torch.int64, device=DEV)
    ops.rollout_random(state, table, k, traj, seed=SEED, step0=3, env_offset=17, action_out=act, stats=stats,
                       uniforms=uniforms)
    torch.cuda.synchronize()
    return [t.clone() for t in (traj.observation, traj.legal_action_mask, traj.rewards, traj.terminated,
                                traj.current_player, act, stats, state)]


@pytest.mark.parametrize("n", [8192, 1001])
@pytest.mark.parametrize("caller_uniforms", [False, True])
def test_rollout_into_compressible_equals_plain(n, caller_uniforms):
    from brl_b200 import ops
    from brl_b200.deals import synthetic_deal_table
    k = 32
    table = torch.as_tensor(synthetic_deal_table(100_000, seed=0), device=DEV)
    state0, out0 = ops.new_state(n, DEV), ops.EnvOutputs(n, DEV)
    ops.init(ops.make_keys(SEED, n, DEV, env_offset=17), table, state0, out0)
    uniforms = None
    if caller_uniforms:
        g = torch.Generator().manual_seed(5)
        uniforms = torch.randint(-2 ** 31, 2 ** 31, (k, n), dtype=torch.int32, generator=g).to(DEV)
    comp = ops.EnvOutputs(n, DEV, rows=k)
    plain = ops.EnvOutputs(n, DEV, rows=k)
    plain.observation = torch.empty_like(comp.observation)
    plain.legal_action_mask = torch.empty_like(comp.legal_action_mask)
    assert comp.observation.shape == (k, n, ops.OBS_DIM) and comp.observation.dtype == torch.float32
    assert comp.observation.is_contiguous() and comp.legal_action_mask.is_contiguous()
    assert comp.legal_action_mask.shape == (k, n, ops.NUM_ACTIONS) and comp.legal_action_mask.dtype == torch.uint8
    names = ("observation", "mask", "rewards", "terminated", "current_player", "action", "stats", "state")
    for name, a, b in zip(names, _rollout(ops, table, state0, plain, k, uniforms), _rollout(ops, table, state0, comp, k, uniforms)):
        assert torch.equal(a, b), name


def test_allocator_returns_memory():
    from brl_b200 import _lib, ops
    L = _lib.load()
    torch.cuda.synchronize()
    gran = L.brl_compressible_granularity(0)
    assert gran > 0
    free0, _ = torch.cuda.mem_get_info()
    # 40 x 8 GB is more than the card holds: a leaked allocation or mapping fails the loop
    for i in range(40):
        buf = _lib.CompressibleBuffer((8 << 30) + 1, 0)
        t = torch.as_tensor(buf, device=DEV)
        assert t.numel() == (8 << 30) + 1
        t[-1] = i
        assert int(t[-1]) == i
        del t, buf
    # the trajectories of EnvOutputs are freed with their last view
    for _ in range(10):
        traj = ops.EnvOutputs(65536, DEV, rows=32)
        obs = traj.observation[1:3]
        del traj
        obs.fill_(1.0)
        del obs
    gc.collect()
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    assert abs(free1 - free0) <= 64 * gran


def test_allocations_are_granularity_multiples_and_aligned():
    from brl_b200 import _lib
    gran = _lib.load().brl_compressible_granularity(0)
    bufs = [_lib.CompressibleBuffer(b, 0) for b in (1, gran - 1, gran, gran + 1, 3 * gran + 5)]
    for b in bufs:
        assert b.ptr % gran == 0
    with pytest.raises(_lib.BrlError):
        _lib.CompressibleBuffer(0, 0)
