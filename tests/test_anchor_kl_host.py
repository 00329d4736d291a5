"""CPU: the KL anchor of PPO -- the float64 reference (tests/anchor_kl_ref.py) against closed forms and finite
differences, the config / population / PBT rules, and the argument checks of the anchored update ops."""
import ctypes
import math

import pytest
import torch

from tests import anchor_kl_ref


def _batch(seed, B=16, A=38):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn((B, A), generator=g, dtype=torch.float64) * 2
    mask = torch.rand((B, A), generator=g) < 0.5
    mask[:, 0] = True
    return g, logits, mask


@pytest.mark.parametrize("masked", [True, False])
def test_anchor_equal_to_policy_gives_zero_kl_and_the_plain_gradient(masked):
    g, logits, mask = _batch(1)
    B = logits.shape[0]
    action = torch.multinomial(mask.double(), 1, generator=g)[:, 0]
    value = torch.randn(B, generator=g, dtype=torch.float64)
    old_lp, old_v, gae, tgt = (torch.randn(B, generator=g, dtype=torch.float64) for _ in range(4))
    kw = dict(clip_eps=0.2, ent_coef=0.01, vf_coef=0.5, masked_policy=masked)
    grads = []
    for anchor in (None, logits.clone()):
        lg = logits.clone().requires_grad_(True)
        total, aux = anchor_kl_ref.loss_fn(lg, value, mask, action, old_lp - 1.0, old_v, gae, tgt, anchor_logits=anchor,
                                           anchor_kl_coef=3.0, **kw)
        total.backward()
        grads.append(lg.grad)
        assert abs(float(aux[-1])) < 1e-14
    assert torch.allclose(grads[0], grads[1], rtol=0, atol=1e-14)


def test_two_actions_match_the_closed_form():
    """pi = (p, 1-p), alpha = (q, 1-q): KL = p log(p/q) + (1-p) log((1-p)/(1-q)), and d KL / d l_0 = p (1-p) (log(p/q) -
    log((1-p)/(1-q))) -- the per-row formula pi_j (log pi_j - log alpha_j - KL) summed with d pi / d l."""
    a = torch.tensor([[0.3, -1.2]], dtype=torch.float64, requires_grad=True)
    anc = torch.tensor([[-0.5, 0.9]], dtype=torch.float64)
    mask = torch.ones((1, 2), dtype=torch.bool)
    kl = anchor_kl_ref.anchor_kl(a, anc, mask)
    kl.backward()
    p = 1 / (1 + math.exp(-(0.3 + 1.2)))
    q = 1 / (1 + math.exp(-(-0.5 - 0.9)))
    want = p * math.log(p / q) + (1 - p) * math.log((1 - p) / (1 - q))
    assert abs(float(kl) - want) < 1e-14
    lr = (math.log(p / q), math.log((1 - p) / (1 - q)))
    want_g = [p * (lr[0] - want), (1 - p) * (lr[1] - want)]  # coef / B * pi_j (log pi_j - log alpha_j - KL), B = 1
    assert torch.allclose(a.grad[0], torch.tensor(want_g, dtype=torch.float64), rtol=0, atol=1e-14)
    assert abs(want_g[0] - p * (1 - p) * (lr[0] - lr[1])) < 1e-14


@pytest.mark.parametrize("masked", [True, False])
def test_gradient_formula_and_finite_differences(masked):
    g, logits, mask = _batch(2, B=6, A=7)
    anchor = torch.randn(logits.shape, generator=g, dtype=torch.float64) * 2
    lg = logits.clone().requires_grad_(True)
    kl = anchor_kl_ref.anchor_kl(lg, anchor, mask, masked)
    kl.backward()
    sel = mask if masked else torch.ones_like(mask)
    neg = torch.tensor(float("-inf"), dtype=torch.float64)
    logp = torch.log_softmax(torch.where(sel, logits, neg), 1)
    loga = torch.log_softmax(torch.where(sel, anchor, neg), 1)
    p = logp.exp()
    d = torch.where(sel, logp - loga, torch.zeros_like(logp))
    kl_b = (p * d).sum(1, keepdim=True)
    want = torch.where(sel, p * (d - kl_b), torch.zeros_like(p)) / logits.shape[0]
    assert torch.allclose(lg.grad, want, rtol=0, atol=1e-14)
    assert not bool(lg.grad[~sel].any())
    assert torch.autograd.gradcheck(lambda x: anchor_kl_ref.anchor_kl(x, anchor, mask, masked), (logits.clone().requires_grad_(True),))


def _config(**kw):
    base = dict(num_envs=64, num_steps=4, minibatch_size=64, update_epochs=1, total_timesteps=64 * 4, hash_size=20, save_model=False)
    base.update(kw)
    return base


@pytest.mark.parametrize("kw,match", [
    (dict(anchor_kl_coef=0.1), "anchor_model_path"),
    (dict(anchor_kl_coef=-0.1, anchor_model_path="anchor.pkl"), "anchor_kl_coef"),
    (dict(anchor_kl_coef=float("nan"), anchor_model_path="anchor.pkl"), "anchor_kl_coef"),
    (dict(anchor_kl_coef=float("inf"), anchor_model_path="anchor.pkl"), "anchor_kl_coef"),
    (dict(anchor_kl_coef="0.1", anchor_model_path="anchor.pkl"), "anchor_kl_coef"),
])
def test_bad_anchor_configs_are_refused_before_any_device_work(kw, match):
    from brl_b200 import ppo
    assert ppo.default_config()["anchor_model_path"] is None and ppo.default_config()["anchor_kl_coef"] == 0.0
    with pytest.raises(ValueError, match=match):
        ppo.train(_config(**kw), 0, device="cpu")
    with pytest.raises(ValueError, match=match):
        ppo.train_population([_config(**kw), _config(seed=1, **kw)], [0, 1], device="cpu")


def test_population_anchors_are_all_or_none():
    from brl_b200 import ppo
    with pytest.raises(ValueError, match="anchor_model_path"):
        ppo.train_population([_config(anchor_model_path="a.pkl", anchor_kl_coef=0.1), _config(seed=1)], [0, 1], device="cpu")


def test_population_update_step_refuses_mixed_anchors():
    from brl_b200.models import make_forward_pass
    from brl_b200.optim import make_optimizer
    from brl_b200.update import make_population_update_step
    cfg = dict(actor_illegal_action_mask=True, clip_eps=0.2, ent_coef=0.0, vf_coef=0.5, num_minibatches=1, minibatch_size=8,
               update_epochs=1, num_steps=2, num_envs=4, lr=1e-3, max_grad_norm=0.5, anneal_lr=False, global_gradient_clipping=True)
    fp = make_forward_pass("relu", "DeepMind")
    step = make_population_update_step([cfg, dict(cfg)], fp, [make_optimizer(cfg), make_optimizer(cfg)])
    assert step.anchor_kl is None
    x = torch.zeros((2, 4))
    with pytest.raises(ValueError, match="anchor_model_path"):
        step([None, None], [None, None], [x, x], [x, x], anchor_logits=[torch.zeros((2, 4, 38)), None])


def test_pbt_may_perturb_the_anchor_coefficient():
    from brl_b200 import pbt
    assert "anchor_kl_coef" in pbt.PERTURBABLE_KEYS
    cfg = pbt.check_pbt_config(dict(perturb_keys=("lr", "anchor_kl_coef")), 2)
    assert cfg["perturb_keys"] == ("lr", "anchor_kl_coef")
    assert pbt.explore({"anchor_kl_coef": 0.5}, {"anchor_kl_coef": 1.25}) == {"anchor_kl_coef": 0.625}


def _bind(L, name):
    fn = getattr(L, name)
    fn.restype, fn.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]
    return fn


def test_anchored_ops_validate_their_arguments_without_a_gpu():
    from brl_b200 import _lib
    L = _lib.load()
    assert L.brl_xla_layout(b"brl_ppo_grad_anchored") == b"iisiiiiiiioosii"
    assert L.brl_xla_layout(b"brl_ppo_grad_grouped_anchored") == b"iiisoosii"
    assert L.brl_xla_layout(b"brl_ppo_grad") == b"iisiiiiiiioos" and L.brl_xla_layout(b"brl_ppo_grad_grouped") == b"iiisoos"
    for name in ("brl_ppo_grad_anchored", "brl_ppo_grad_grouped_anchored"):
        assert name in _lib.OPS and name in _lib.LAZY_OPS and name + "_xla" in _lib.XLA_LEGACY
    solo, grouped = _bind(L, "brl_ppo_grad_anchored"), _bind(L, "brl_ppo_grad_grouped_anchored")
    fake = lambda n: (ctypes.c_void_p * n)(*[ctypes.c_void_p(4096)] * n)  # noqa: E731 -- never dereferenced
    pp = _lib.BrlPpoParams(1024, 4096, 0.2, 0.01, 0.5, 0.0, _lib.PPO_VALUE_CLIPPING, 0)
    assert solo(None, fake(15), ctypes.byref(pp), 8) == -1 and b"BrlPpoParams" in L.brl_last_error()
    assert solo(None, (ctypes.c_void_p * 15)(), ctypes.byref(pp), ctypes.sizeof(pp)) == -2 and b"'obs' is NULL" in L.brl_last_error()
    for k, name in ((13, b"anchor_logits"), (14, b"kl_coef")):
        b = fake(15)
        b[k] = None
        assert solo(None, b, ctypes.byref(pp), ctypes.sizeof(pp)) == -2
        assert b"brl_ppo_grad_anchored: buffer '" + name + b"' is NULL" in L.brl_last_error()
    pp.batch = -1
    assert solo(None, fake(15), ctypes.byref(pp), ctypes.sizeof(pp)) == -1 and b"batch" in L.brl_last_error()
    pp.batch = 0  # an empty batch is a no-op: NULL buffers are never looked at
    assert solo(None, (ctypes.c_void_p * 15)(), ctypes.byref(pp), ctypes.sizeof(pp)) == 0
    gp = _lib.BrlPpoGroupedParams(1024, 3, 0, 0, 0)
    assert grouped(None, fake(9), ctypes.byref(gp), 4) == -1 and b"BrlPpoGroupedParams" in L.brl_last_error()
    for k, name in ((7, b"anchor_logits"), (8, b"kl_coef")):
        b = fake(9)
        b[k] = None
        assert grouped(None, b, ctypes.byref(gp), ctypes.sizeof(gp)) == -2
        assert b"brl_ppo_grad_grouped_anchored: buffer '" + name + b"' is NULL" in L.brl_last_error()
    for batch, K in ((0, 3), (1024, 0)):
        gp.batch, gp.n_learners = batch, K
        assert grouped(None, (ctypes.c_void_p * 9)(), ctypes.byref(gp), ctypes.sizeof(gp)) == 0
    gp.n_learners = _lib.MAX_LEARNERS + 1
    assert grouped(None, fake(9), ctypes.byref(gp), ctypes.sizeof(gp)) == -1 and b"n_learners" in L.brl_last_error()


def test_ops_keywords_go_together():
    from brl_b200 import _lib, ops
    with pytest.raises(_lib.BrlError, match="together"):
        ops._anchor_args("ppo_grad", torch.zeros(1), None)
    with pytest.raises(_lib.BrlError, match="together"):
        ops._anchor_args("ppo_grad_grouped", None, torch.zeros(1))
