"""CPU: call-value policy improvement (DESIGN.md f17).  The float64 restatement of brl_cv_grad's loss (tests/cvi_ref.py)
on hand-worked cases and against central finite differences, the ops' registration and XLA layouts, and cvi.train's
config checks, which must fire before any CUDA call."""
import math
import pickle

import numpy as np
import pytest

from tests import cvi_ref as R

NAN = float("nan")


def _row(pairs):
    """a [1, 38] gain row with the given {call: gain}, NaN elsewhere"""
    g = np.full((1, 38), NAN)
    for a, x in pairs.items():
        g[0, a] = x
    return g


def test_two_legal_calls_at_equal_logits():
    g = _row({0: 3.0, 5: -1.0})
    lg = np.zeros((1, 38))
    loss, grad, st = R.loss_grad_stats(lg, g, 0.0)
    # pi = (1/2, 1/2): gbar = 1, J = 1 / 24
    assert math.isclose(st[1], 1.0) and math.isclose(loss, -1.0 / 24)
    # d loss / d l_0 = -1/2 (3 - 1) / 24, d / d l_5 = -1/2 (-1 - 1) / 24
    assert math.isclose(grad[0, 0], -1.0 / 24) and math.isclose(grad[0, 5], 1.0 / 24)
    assert (grad[0, [a for a in range(38) if a not in (0, 5)]] == 0).all()
    # ties in the logits: the lowest index (0, gain 3, the best call)
    assert st[2] == 3.0 and st[3] == 0.0 and st[5] == 1.0
    assert math.isclose(st[4], math.log(2))
    assert math.isclose(st[6], 36 / 38)                 # the unmasked softmax puts 1/38 on each call


def test_equal_gains_give_no_policy_gradient():
    rng = np.random.default_rng(1)
    lg = rng.normal(size=(5, 38))
    g = np.where(rng.random((5, 38)) < 0.5, 2.0, NAN)
    g[:, 0] = 2.0
    loss, grad, st = R.loss_grad_stats(lg, g, 0.0)
    assert np.abs(grad).max() < 1e-15
    assert math.isclose(st[1], 2.0) and st[3] == 0.0 and st[5] == 1.0


def test_single_legal_call():
    g = _row({7: -5.0})
    lg = np.random.default_rng(2).normal(size=(1, 38))
    loss, grad, st = R.loss_grad_stats(lg, g, 0.1)
    assert (grad == 0).all()
    assert st[4] == 0.0 and st[1] == -5.0 and st[2] == -5.0 and st[3] == 0.0 and st[5] == 1.0
    assert math.isclose(loss, 5.0 / 24)


def test_illegal_entries_are_ignored():
    rng = np.random.default_rng(3)
    lg = rng.normal(size=(4, 38))
    g = np.where(rng.random((4, 38)) < 0.4, rng.integers(-10, 10, (4, 38)).astype(float), NAN)
    g[:, 1] = 1.0
    _, grad, st = R.loss_grad_stats(lg, g, 0.05)
    lg2 = np.where(np.isfinite(g), lg, lg + rng.normal(size=lg.shape) * 5)   # moving an illegal logit changes nothing legal
    _, grad2, st2 = R.loss_grad_stats(lg2, g, 0.05)
    assert np.allclose(grad, grad2, atol=1e-15) and np.allclose(st[:6], st2[:6])
    assert (grad[~np.isfinite(g)] == 0).all()


def test_ties_in_the_argmax_statistics():
    g = _row({0: 1.0, 3: 4.0, 9: 4.0})
    lg = np.full((1, 38), -1.0)
    lg[0, [3, 9]] = 2.0                                  # 3 and 9 tie on the logit: 3, a best call
    _, _, st = R.loss_grad_stats(lg, g, 0.0)
    assert st[2] == 4.0 and st[3] == 0.0 and st[5] == 1.0
    lg[0, 0] = 2.0                                       # now 0 ties too and wins: gain 1, regret 3
    _, _, st = R.loss_grad_stats(lg, g, 0.0)
    assert st[2] == 1.0 and st[3] == 3.0 and st[5] == 0.0
    g[0, 0] = 4.0                                        # ties in the gains: the argmax call is one of the best
    _, _, st = R.loss_grad_stats(lg, g, 0.0)
    assert st[5] == 1.0


def test_no_legal_call_adds_only_illegal_mass():
    g = np.full((2, 38), NAN)
    g[1, 4] = 6.0
    lg = np.zeros((2, 38))
    _, grad, st = R.loss_grad_stats(lg, g, 0.1)
    assert (grad[0] == 0).all()
    assert math.isclose(st[1], 3.0) and math.isclose(st[6], (1.0 + 37 / 38) / 2) and st[5] == 0.5


@pytest.mark.parametrize("ent", [0.0, 0.03])
def test_finite_differences_match_the_gradient(ent):
    rng = np.random.default_rng(4)
    B = 6
    lg = rng.normal(size=(B, 38))
    g = np.where(rng.random((B, 38)) < 0.5, rng.integers(-20, 20, (B, 38)).astype(float), NAN)
    g[:, 0] = 0.0
    _, grad, _ = R.loss_grad_stats(lg, g, ent)
    h = 1e-6
    for b, j in [(b, j) for b in range(B) for j in range(38)]:
        up, dn = lg.copy(), lg.copy()
        up[b, j] += h
        dn[b, j] -= h
        fd = (R.loss_grad_stats(up, g, ent)[0] - R.loss_grad_stats(dn, g, ent)[0]) / (2 * h)
        assert abs(fd - grad[b, j]) < 1e-8, (b, j, fd, grad[b, j])


def test_torch_loss_equals_the_numpy_restatement():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(5)
    lg = rng.normal(size=(7, 38))
    g = np.where(rng.random((7, 38)) < 0.5, rng.integers(-20, 20, (7, 38)).astype(float), NAN)
    g[:, 2] = 1.0
    t = torch.tensor(lg, requires_grad=True)
    loss = R.torch_loss(t, torch.tensor(g), 0.02)
    loss.backward()
    want, grad, _ = R.loss_grad_stats(lg, g, 0.02)
    assert math.isclose(float(loss.detach()), want, rel_tol=1e-12)
    assert np.allclose(t.grad.numpy(), grad, atol=1e-14)


def test_ops_are_registered_with_xla_layouts():
    from brl_b200 import _lib
    for op, layout in (("brl_cv_grad", b"iisioos"), ("brl_cv_eval", b"iisios")):
        assert op in _lib.OPS and op in _lib.LAZY_OPS and op + "_xla" in _lib.XLA_LEGACY
    L = _lib.load()
    assert L.brl_xla_layout(b"brl_cv_grad") == b"iisioos" and L.brl_xla_layout(b"brl_cv_eval") == b"iisios"
    assert L.brl_xla_layout(b"brl_call_values") == b"iiiiiisoooooooooooo"   # the examples [19] / [20] are NULL there


def _no_cuda(monkeypatch):
    import torch

    def boom(*a, **k):
        raise AssertionError("CUDA touched before the config was checked")
    for name in ("synchronize", "current_stream", "set_device"):
        monkeypatch.setattr(torch.cuda, name, boom)
    from brl_b200 import cvi, env
    monkeypatch.setattr(env, "BridgeBidding", boom)
    monkeypatch.setattr(cvi, "BridgeBidding", boom)
    monkeypatch.setattr(cvi, "init_params", boom)
    monkeypatch.setattr(cvi, "load_params", boom)


BAD = [dict(boards_per_iter=0), dict(num_iters=-1), dict(epochs=0), dict(minibatch_size=0), dict(num_eval_envs=0),
       dict(num_eval_step=0), dict(save_model_interval=0), dict(minibatch_size=1.5), dict(ent_coef=-0.1),
       dict(ent_coef=float("nan")), dict(lr=float("inf")), dict(lr=-1e-6), dict(max_grad_norm=-1.0), dict(bogus=1)]


@pytest.mark.parametrize("bad", BAD, ids=lambda d: "-".join(f"{k}={v}" for k, v in d.items()))
def test_config_errors_fire_before_any_device_work(bad, monkeypatch):
    from brl_b200 import cvi
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError):
        cvi.train(bad, 0, np.zeros((10, 48), np.uint8), device="cuda")


@pytest.mark.parametrize("key", ["initial_model_path", "opponent_model_path", "eval_opp_model_path"])
def test_a_model_file_that_is_not_a_deepmind_net_is_refused(key, tmp_path, monkeypatch):
    from brl_b200 import cvi
    p = tmp_path / "bad.pkl"
    p.write_bytes(pickle.dumps({"actor_critic/linear": {"w": np.zeros((3, 3)), "b": np.zeros(3)}}))
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError, match="DeepMind"):
        cvi.train({key: str(p)}, 0, np.zeros((10, 48), np.uint8))


def test_a_process_group_of_several_ranks_is_refused(monkeypatch):
    from brl_b200 import cvi, dist
    monkeypatch.setattr(dist, "rank_world", lambda: (0, 2))
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError, match="one GPU"):
        cvi.train({}, 0, np.zeros((10, 48), np.uint8))


def test_keys_and_permutations_depend_on_seed_and_iteration():
    import torch
    from brl_b200 import cvi
    keys = {cvi.iteration_key(s, i) for s in range(3) for i in range(50)}
    assert len(keys) == 150
    a = torch.randperm(100, generator=cvi.permutation_generator(1, 2))
    b = torch.randperm(100, generator=cvi.permutation_generator(1, 2))
    c = torch.randperm(100, generator=cvi.permutation_generator(1, 3))
    assert torch.equal(a, b) and not torch.equal(a, c)
