"""GPU: brl_duplicate_match, a whole duplicate match as one device-resident call -- bit-equal to the host loop of
make_simple_duplicate_evaluate, the golden seeded match, capture in a CUDA graph, the graph cache, the XLA symbol, the bad-net
status and the empty batch.  The self-play league on this op is checked against pairwise host matches in test_cuda_league."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import helpers as H
from tests.test_cuda_xla import _call_xla

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FORCE_FUSED, FORCE_LAYERS = 1 << 30, 1 << 29  # BRL_F_TUNE_MLP_FUSED, BRL_F_TUNE_MLP_LAYERS (include/brl_b200.h)


def _env(rows=5000, seed=4):
    from brl_b200 import BridgeBidding
    from brl_b200.deals import synthetic_deal_table
    return BridgeBidding(table=synthetic_deal_table(rows, seed=seed), device=DEV)


def _pin_host_path(monkeypatch, tune):
    """make the host loop's per-team listed forwards take the path `tune` pins"""
    from brl_b200 import ops
    orig = ops.policy_act_rows
    monkeypatch.setattr(ops, "policy_act_rows", lambda *a, **kw: orig(*a, **{**kw, "tune": kw.get("tune", 0) | tune}))


def _compare_two_team(env, n, key_seed, tune=0):
    from brl_b200 import random as brandom
    from brl_b200.evaluation import make_device_duplicate_evaluate, make_simple_duplicate_evaluate
    nets = [H.seeded_params(600, DEV), H.seeded_params(601, DEV)]
    key = brandom.PRNGKey(key_seed)
    want = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)(nets[0], nets[1], key)
    got = make_device_duplicate_evaluate(env, "relu", "DeepMind", n, tune=tune)(nets[0], nets[1], key)
    np.testing.assert_allclose(got[0], want[0], rtol=1e-12, atol=0)
    for t_got, t_want in zip(got[1:3], want[1:3]):
        for f in t_want._fields:
            assert torch.equal(getattr(t_got, f), getattr(t_want, f)), f
    assert torch.equal(got[3], want[3])


@pytest.mark.parametrize("n", [1, 100, 257, 1000])
def test_device_match_equals_the_two_team_host_loop(n):
    _compare_two_team(_env(), n, key_seed=n)


@pytest.mark.parametrize("tune", [FORCE_LAYERS, FORCE_FUSED])
@pytest.mark.parametrize("n", [4096 + 77, 65536])
def test_device_match_equals_the_host_loop_on_a_pinned_path(n, tune, monkeypatch):
    _pin_host_path(monkeypatch, tune)
    _compare_two_team(_env(), n, key_seed=3, tune=tune)


def test_device_match_reproduces_the_golden_seeded_match():
    from brl_b200 import BridgeBidding, random as brandom
    from brl_b200.evaluation import make_device_duplicate_evaluate
    g = H.load_c1_seeded()
    env = BridgeBidding(table=H.load_boards()["table"], device=DEV)
    nets = [H.seeded_params(int(s), DEV) for s in g["weight_seeds"]]
    log, _, _, cum = make_device_duplicate_evaluate(env, "relu", "DeepMind", int(g["n"]))(nets[0], nets[1],
                                                                                        brandom.PRNGKey(int(g["seed"])))
    assert (cum.cpu().numpy() == g["imps"]).all()
    np.testing.assert_allclose(log, g["stats"], rtol=1e-9, atol=1e-12)   # IMP, SE, win rate


class _Match:
    """one two-net match's buffers and a direct call"""

    def __init__(self, n=700, seed=5):
        from brl_b200 import ops
        from brl_b200.models import make_forward_pass
        self.env = _env(3000, seed=seed)
        self.n = n
        self.keys = ops.make_keys(seed, n, DEV)
        self.pool = ops.mlp_pack_pool([H.seeded_params(700, DEV), H.seeded_params(701, DEV)], make_forward_pass().pack_into)
        self.scratch = torch.empty(ops.duplicate_match_scratch_bytes(n, 2), dtype=torch.uint8, device=DEV)

    def outputs(self):
        from brl_b200 import ops
        return dict(cum_return=torch.full((self.n,), 9.0, device=DEV), sums=torch.zeros(8, dtype=torch.float64, device=DEV),
                    status=torch.full((1,), 7, dtype=torch.int32, device=DEV),
                    table_a=ops.TableInfoBuffers(self.n, DEV), table_b=ops.TableInfoBuffers(self.n, DEV))

    def call(self, out, **kw):
        from brl_b200 import ops
        ops.duplicate_match(self.keys, self.env.table, self.pool, self.scratch, out["cum_return"], out["sums"], out["status"],
                            table_a=out["table_a"], table_b=out["table_b"], **kw)


def _flat(out):
    return ([out["cum_return"], out["sums"], out["status"]] + [getattr(out["table_a"], k) for k in out["table_a"].__slots__] +
            [getattr(out["table_b"], k) for k in out["table_b"].__slots__])


@pytest.mark.parametrize("capture_error_mode", ["global", "thread_local"])
def test_captured_in_a_cuda_graph_and_cached(capture_error_mode):
    """inside torch.cuda.graph the op adds its loop to the caller's capture: it cannot synchronise with the host there, and
    both replays equal a direct call.  A second direct call with the same buffers relaunches the cached graph."""
    from brl_b200 import ops
    m = _Match()
    ref = m.outputs()
    m.call(ref)
    torch.cuda.synchronize()
    assert int(ref["status"][0]) == 0 and float(ref["sums"][0]) == m.n
    again = m.outputs()
    m.call(again)   # other output buffers: a graph of their own (unless the allocator handed back ref's addresses)
    builds = ops.duplicate_match_graph_builds()
    again["sums"].zero_()
    m.call(again)   # the same buffers: the cached graph is relaunched
    torch.cuda.synchronize()
    assert ops.duplicate_match_graph_builds() == builds
    for a, b in zip(_flat(again), _flat(ref)):
        assert torch.equal(a, b)
    out = m.outputs()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, capture_error_mode=capture_error_mode):
        out["sums"].zero_()
        m.call(out)
    assert ops.duplicate_match_graph_builds() == builds   # the capture builds nothing of its own
    for _ in range(2):
        for t in _flat(out):
            t.fill_(3)
        g.replay()
        torch.cuda.synchronize()
        for a, b in zip(_flat(out), _flat(ref)):
            assert torch.equal(a, b)


def test_xla_symbol_equals_the_direct_call():
    from brl_b200 import ops
    m = _Match(n=513, seed=6)
    ref = m.outputs()
    m.call(ref)
    out = m.outputs()
    tensors = [m.keys, m.env.table, m.pool, None, None, m.scratch, out["cum_return"], out["sums"], out["status"]] + \
        [getattr(out["table_a"], k) for k in out["table_a"].__slots__] + [getattr(out["table_b"], k) for k in out["table_b"].__slots__]
    _call_xla("brl_duplicate_match", tensors, ops._params(m.n, k_steps=2, n_deals=m.env.table.shape[0]))
    torch.cuda.synchronize()
    for a, b in zip(_flat(out), _flat(ref)):
        assert torch.equal(a, b)


def test_a_bad_net_id_stops_the_loop_with_a_status_and_an_empty_batch_is_a_no_op():
    from brl_b200 import _lib, ops
    from brl_b200.evaluation import _check_match_status
    m = _Match(n=300, seed=7)
    M = 2
    env_models = torch.zeros((m.n, 2), dtype=torch.int32, device=DEV)
    env_models[:, 1] = 1
    env_models[17] = M                      # both seats of env 17 name a net outside the pool
    out = m.outputs()
    ops.duplicate_match(m.keys, m.env.table, m.pool, m.scratch, out["cum_return"], out["sums"], out["status"],
                        env_models=env_models)
    torch.cuda.synchronize()
    assert int(out["status"][0]) == _lib.MATCH_BAD_MODEL
    with pytest.raises(_lib.BrlError, match="outside"):
        _check_match_status(int(out["status"][0]))
    env_models[17] = torch.tensor([0, 1], dtype=torch.int32, device=DEV)   # the same buffers, valid again
    ops.duplicate_match(m.keys, m.env.table, m.pool, m.scratch, out["cum_return"], out["sums"], out["status"],
                        env_models=env_models)
    torch.cuda.synchronize()
    assert int(out["status"][0]) == _lib.MATCH_OK
    L = _lib.load()
    nulls = (C.c_void_p * 21)()
    p0 = ops._params(0, k_steps=3)
    assert L.brl_duplicate_match(C.c_void_p(torch.cuda.current_stream().cuda_stream), nulls, C.byref(p0), C.sizeof(p0)) == 0
    torch.cuda.synchronize()
