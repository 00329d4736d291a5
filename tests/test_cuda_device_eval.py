"""GPU: brl_evaluate_match, make_evaluate / make_simple_evaluate as one device-resident call -- equal to their host loops per
env and in every statistic, the golden seeded match, the graph cache, capture in a CUDA graph, ppo.train with the device
evaluators against the same run with the host loops, and the XLA symbol."""
import numpy as np
import pytest
import torch

from tests import helpers as H
from tests.test_cuda_xla import _call_xla

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _env(rows=5000, seed=4):
    from brl_b200 import BridgeBidding
    from brl_b200.deals import synthetic_deal_table
    return BridgeBidding(table=synthetic_deal_table(rows, seed=seed), device=DEV)


@pytest.fixture
def precision(request, monkeypatch):
    """every forward pass the evaluators make runs in `request.param`"""
    import brl_b200.evaluation as ev
    orig = ev.make_forward_pass
    monkeypatch.setattr(ev, "make_forward_pass", lambda **kw: orig(precision=request.param, **kw))
    return request.param


def _host_acc(monkeypatch):
    """the host loop's per-env acc rows and cum_return, as handed to eval_summary"""
    from brl_b200 import ops
    seen = {}
    orig = ops.eval_summary

    def spy(acc, cum_return, *a, **kw):
        seen["acc"], seen["cum_return"] = acc.clone(), cum_return.clone()
        return orig(acc, cum_return, *a, **kw)
    monkeypatch.setattr(ops, "eval_summary", spy)
    return seen


def _assert_log_info(got, want):
    assert len(got) == len(want)
    for g, w in zip(got, want):  # f64 sums formed with atomics: the last bits may move
        np.testing.assert_allclose(np.asarray(g, dtype=np.float64), np.asarray(w, dtype=np.float64), rtol=1e-12, atol=0)


SIZES = [1, 100, 4095, 4097, 10000]   # padded live rows on both sides of the fused forward's 4096


@pytest.mark.parametrize("precision", ["tc", "tc-bf16"], indirect=True)
@pytest.mark.parametrize("game_mode", ["competitive", "free-run"])
@pytest.mark.parametrize("n", SIZES)
def test_device_duplicate_evaluate_equals_the_host_loop(n, game_mode, precision, monkeypatch):
    from brl_b200 import random as brandom
    from brl_b200.evaluation import make_device_evaluate, make_evaluate, make_evaluate_log
    env = _env()
    actor, opp = H.seeded_params(800, DEV), H.seeded_params(801, DEV)
    key = brandom.PRNGKey(20 + n)
    seen = _host_acc(monkeypatch)
    want = make_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, game_mode, duplicate=True,
                         team2_params=opp)(actor, key)
    dev_eval = make_device_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, game_mode, duplicate=True,
                                    team2_params=opp)
    got = dev_eval(actor, key)
    assert torch.equal(dev_eval.buffers.acc, seen["acc"])
    assert torch.equal(dev_eval.buffers.cum_return, seen["cum_return"])
    for t_got, t_want in zip(got[1:], want[1:]):
        for f in t_want._fields:
            assert torch.equal(getattr(t_got, f), getattr(t_want, f)), f
    _assert_log_info(got[0], want[0])
    assert list(make_evaluate_log(got[0])) == list(make_evaluate_log(want[0]))


@pytest.mark.parametrize("precision", ["tc", "tc-bf16"], indirect=True)
@pytest.mark.parametrize("game_mode", ["competitive", "free-run"])
@pytest.mark.parametrize("n", SIZES)
def test_device_single_table_evaluate_equals_the_host_loop(n, game_mode, precision, monkeypatch):
    from brl_b200 import random as brandom
    from brl_b200.evaluation import make_device_evaluate, make_evaluate
    env = _env()
    actor, opp = H.seeded_params(810, DEV), H.seeded_params(811, DEV)
    key = brandom.PRNGKey(40 + n)
    seen = _host_acc(monkeypatch)
    want_state, want_log = make_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, game_mode,
                                         team2_params=opp)(actor, key)
    dev_eval = make_device_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, game_mode, team2_params=opp)
    got_state, got_log = dev_eval(actor, key)
    assert torch.equal(dev_eval.buffers.acc, seen["acc"])
    assert torch.equal(dev_eval.buffers.cum_return, seen["cum_return"])
    assert torch.equal(got_state._packed, want_state._packed)
    assert torch.equal(got_state.rewards, want_state.rewards)   # the summed step rewards
    for k in ("observation", "_mask_u8", "_terminated_u8", "current_player"):
        assert torch.equal(getattr(got_state, k), getattr(want_state, k)), k
    _assert_log_info(got_log, want_log)


@pytest.mark.parametrize("precision", ["tc", "tc-bf16"], indirect=True)
@pytest.mark.parametrize("n, seed", [(1, 0), (300, 1), (4097, 2), (10000, 3)])
def test_device_simple_evaluate_equals_the_host_loop(n, seed, precision):
    from brl_b200 import random as brandom
    from brl_b200.evaluation import make_device_simple_evaluate, make_simple_evaluate
    env = _env()
    actor, opp = H.seeded_params(820 + seed, DEV), H.seeded_params(830 + seed, DEV)
    key = brandom.PRNGKey(60 + seed)
    trace = []
    want = make_simple_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, team2_params=opp)(actor, key, trace=trace)
    dev_eval = make_device_simple_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, team2_params=opp)
    got = dev_eval(actor, key)
    assert trace[-1][0] == "R" and torch.equal(dev_eval.buffers.cum_return, trace[-1][1])
    assert float(got) == float(want)


def test_device_evaluate_reproduces_the_golden_seeded_match(monkeypatch):
    from brl_b200 import BridgeBidding, random as brandom
    from brl_b200.evaluation import make_device_evaluate, make_evaluate
    g = H.load_c1_seeded()
    env = BridgeBidding(table=H.load_boards()["table"], device=DEV)
    nets = [H.seeded_params(int(s), DEV) for s in g["weight_seeds"]]
    n, key = int(g["n"]), brandom.PRNGKey(int(g["seed"]))
    args = (env, "relu", "DeepMind", "relu", "DeepMind", None, n, "competitive")
    want = make_evaluate(*args, duplicate=True, team2_params=nets[1])(nets[0], key)
    dev_eval = make_device_evaluate(*args, duplicate=True, team2_params=nets[1])
    got = dev_eval(nets[0], key)
    _assert_log_info(got[0], want[0])
    assert (dev_eval.buffers.cum_return.cpu().numpy() == g["imps"]).all()
    np.testing.assert_allclose(got[0][0], g["stats"][0], rtol=1e-9, atol=1e-12)   # IMP_reward = the golden match's IMP


class _Eval:
    """one duplicate evaluation's buffers and a direct call"""

    def __init__(self, n=700, seed=5):
        from brl_b200 import ops
        from brl_b200.models import make_forward_pass
        self.env = _env(3000, seed=seed)
        self.n = n
        self.keys = ops.make_keys(seed, n, DEV)
        self.pool = ops.mlp_pack_pool([H.seeded_params(900, DEV), H.seeded_params(901, DEV)], make_forward_pass().pack_into)
        self.scratch = torch.empty(ops.evaluate_match_scratch_bytes(n, 1), dtype=torch.uint8, device=DEV)

    def outputs(self):
        from brl_b200 import _lib, ops
        return dict(cum_return=torch.full((self.n,), 9.0, device=DEV),
                    acc=torch.full((self.n, _lib.EVAL_ACC_COLS), 5.0, device=DEV),
                    sums=torch.zeros(_lib.load().brl_eval_num_sums(), dtype=torch.float64, device=DEV),
                    status=torch.full((1,), 7, dtype=torch.int32, device=DEV),
                    table_a=ops.TableInfoBuffers(self.n, DEV), table_b=ops.TableInfoBuffers(self.n, DEV))

    def call(self, out, **kw):
        from brl_b200 import _lib, ops
        ops.evaluate_match(self.keys, self.env.table, self.pool, self.scratch, out["cum_return"], out["status"],
                           mode=_lib.EVAL_MATCH_DUPLICATE, acc=out["acc"], sums=out["sums"], table_a=out["table_a"],
                           table_b=out["table_b"], **kw)


def _flat(out):
    return ([out["cum_return"], out["acc"], out["status"]] + [getattr(out["table_a"], k) for k in out["table_a"].__slots__] +
            [getattr(out["table_b"], k) for k in out["table_b"].__slots__])


def _same(got, want):
    for a, b in zip(_flat(got), _flat(want)):
        assert torch.equal(a, b)
    np.testing.assert_allclose(got["sums"].cpu().numpy(), want["sums"].cpu().numpy(), rtol=1e-12, atol=0)


def test_repeated_calls_relaunch_the_cached_graph():
    """the device twin's second call, with new params and a new key, relaunches the graph its first call built"""
    from brl_b200 import ops, random as brandom
    from brl_b200.evaluation import make_device_evaluate, make_evaluate
    env = _env()
    opp = H.seeded_params(911, DEV)
    args = (env, "relu", "DeepMind", "relu", "DeepMind", None, 2000, "competitive")
    dev_eval = make_device_evaluate(*args, duplicate=True, team2_params=opp)
    dev_eval(H.seeded_params(910, DEV), brandom.PRNGKey(1))
    builds = ops.duplicate_match_graph_builds()
    actor, key = H.seeded_params(912, DEV), brandom.PRNGKey(2)
    got = dev_eval(actor, key)
    assert ops.duplicate_match_graph_builds() == builds
    want = make_evaluate(*args, duplicate=True, team2_params=opp)(actor, key)
    _assert_log_info(got[0], want[0])


@pytest.mark.parametrize("capture_error_mode", ["global", "thread_local"])
def test_captured_in_a_cuda_graph(capture_error_mode):
    """inside torch.cuda.graph the op adds its loop to the caller's capture; both replays equal a direct call"""
    from brl_b200 import ops
    m = _Eval()
    ref = m.outputs()
    m.call(ref)
    torch.cuda.synchronize()
    assert int(ref["status"][0]) == 0 and float(ref["sums"][0]) == m.n
    builds = ops.duplicate_match_graph_builds()
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
        _same(out, ref)


def test_xla_symbol_equals_the_direct_call():
    from brl_b200 import _lib, ops
    m = _Eval(n=513, seed=6)
    ref = m.outputs()
    m.call(ref)
    out = m.outputs()
    tensors = [m.keys, m.env.table, m.pool, m.scratch, out["cum_return"], out["acc"], out["sums"], out["status"]] + \
        [getattr(out["table_a"], k) for k in out["table_a"].__slots__] + \
        [getattr(out["table_b"], k) for k in out["table_b"].__slots__] + [None] * 6
    _call_xla("brl_evaluate_match", tensors,
              ops._params(m.n, n_deals=m.env.table.shape[0], flags=_lib.f_eval_match(_lib.EVAL_MATCH_DUPLICATE)))
    torch.cuda.synchronize()
    _same(out, ref)


def test_ppo_train_with_the_device_evaluators_equals_the_host_evaluators(monkeypatch):
    from brl_b200 import ppo, random as brandom
    from brl_b200.deals import synthetic_deal_table
    from brl_b200.models import params_to_numpy
    config = dict(num_envs=256, num_steps=4, minibatch_size=256, update_epochs=1, total_timesteps=256 * 4 * 3,
                  num_eval_envs=512, num_prioritized_envs=100, num_eval_step=1, self_play=True, ratio_model_zoo=1.0,
                  prioritized_fictitious=True, lr=1e-4, save_model=False)

    def run():
        return ppo.train(config, brandom.PRNGKey(0), tables=[synthetic_deal_table(300, seed=k) for k in range(2)],
                         eval_table=synthetic_deal_table(400, seed=9), device=DEV, eval_opp_params=H.seeded_params(950, DEV))
    with monkeypatch.context() as m:   # the host loops, with the host-list zoo and its one match per model
        m.setattr(ppo, "make_evaluators", H.host_evaluators)
        m.setattr(ppo, "device_zoo_fits", lambda *a, **kw: False)
        host_runner, host_logs = run()
    dev_runner, dev_logs = run()
    assert len(host_logs) == len(dev_logs) == 3
    for h, d in zip(host_logs, dev_logs):
        keys = [k for k in h if k.startswith(("train/score", "train/imp_opp", "eval/"))]
        assert "eval/IMP_reward" in keys and "train/imp_opp_before" in keys
        assert sorted(keys) == sorted(k for k in d if k.startswith(("train/score", "train/imp_opp", "eval/")))
        for k in keys:
            np.testing.assert_allclose(d[k], h[k], rtol=1e-12, atol=0, err_msg=k)
    a, b = params_to_numpy(dev_runner[0]), params_to_numpy(host_runner[0])
    assert all((a[k] == b[k]).all() for k in a)
