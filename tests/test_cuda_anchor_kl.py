"""GPU: the KL anchor of PPO -- brl_ppo_grad_anchored against float64 autograd of the restated loss plus KL
(tests/anchor_kl_ref.py), its coefficient-0 and grouped bit-identities, the roll-out's anchor logits, and ppo.train /
train_population with anchors."""
import numpy as np
import pytest
import torch

from tests import anchor_kl_ref
from tests.test_cuda_population import _COEFS, _bits, _learner, _row

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _anchor_rows(seed, total):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn((total, 38), generator=g) * 1.5).to(DEV).contiguous()


def _call(t, blob, B, coef, *, anchor=None, kl=None, scratch=None, tune=0, **cfg):
    """one ppo_grad (anchored when `anchor` is given) -> (grads, stats, acc)"""
    from brl_b200 import ops
    n = ops.mlp_num_params()
    grads = torch.full((n,), float("nan"), device=DEV)
    stats = torch.full((8,), float("nan"), device=DEV)
    acc = torch.empty(ops.ppo_scratch(DEV).shape, dtype=torch.float64, device=DEV)
    acc.view(torch.uint8).fill_(0xFF)
    if scratch is None:
        scratch = torch.full((int(ops._lib.load().brl_mlp_train_scratch_bytes(B)),), 0xFF, dtype=torch.uint8, device=DEV)
    kw = {} if anchor is None else dict(anchor_logits=anchor, kl_coef=torch.tensor([kl], dtype=torch.float32, device=DEV))
    ops.ppo_grad(t["obs"], blob, scratch, t["index"], t["mask"], t["action"], t["old_lp"], t["old_v"], t["adv"], t["tgt"], grads,
                 stats, acc, clip_eps=coef[0], ent_coef=coef[1], vf_coef=coef[2], illegal_l2_coef=coef[3], tune=tune, **cfg, **kw)
    torch.cuda.synchronize()
    return grads, stats, acc


@pytest.mark.parametrize("B,tune,masked,obs_dtype", [
    (1000, 0, True, torch.uint8),
    (8205, 4 | 16, False, torch.bfloat16),   # the other tile widths, the unmasked policy, ragged row tiles
    (1024, 16, True, torch.float32),
])
def test_ppo_grad_anchored_matches_float64_autograd(B, tune, masked, obs_dtype):
    from brl_b200 import ops
    from brl_b200.models import params_to_numpy
    from brl_b200.optim import flatten_params
    total = 3 * B
    params, t = _learner(51, total, B, obs_dtype)
    obs = t["obs"].cpu().double()
    # rows whose hidden pre-activations stay 2e-5 from zero in float64 (the ReLU kink, as in test_cuda_ppo.py)
    pn = {k: torch.tensor(v, dtype=torch.float64) for k, v in params_to_numpy(params).items()}
    h, margin = obs, torch.full((total,), float("inf"), dtype=torch.float64)
    for i in range(4):
        z = h @ pn[f"w{i}"] + pn[f"b{i}"]
        margin = torch.minimum(margin, z.abs().min(dim=1).values)
        h = torch.relu(z)
    safe = torch.nonzero(margin > 2e-5)[:, 0]
    assert len(safe) >= B
    g = torch.Generator().manual_seed(6)
    idx = safe[torch.randperm(len(safe), generator=g)[:B]]
    t["index"] = idx.to(torch.int32).to(DEV)
    mask, action = t["mask"].cpu().bool(), t["action"].cpu()
    ref = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in params_to_numpy(params).items()}
    hs, zs = [obs[idx]], []
    for i in range(4):
        z = hs[-1] @ ref[f"w{i}"] + ref[f"b{i}"]
        z.retain_grad()
        zs.append(z)
        hs.append(torch.relu(z))
    lg = hs[-1] @ ref["w4"] + ref["b4"]
    vl = (hs[-1] @ ref["w5"] + ref["b5"])[:, 0]
    lg.retain_grad()
    vl.retain_grad()
    old_lp, old_v, tgt, adv = (t[k].cpu().double() for k in ("old_lp", "old_v", "tgt", "adv"))
    anchor = _anchor_rows(7, total).cpu()
    with torch.no_grad():  # old log-probs near the current policy; an anchor near it too, so that KL is moderate
        pl = torch.where(mask[idx], lg, torch.tensor(float("-inf"), dtype=torch.float64)) if masked else lg
        old_lp[idx] = torch.log_softmax(pl, 1).gather(1, action[idx].long()[:, None])[:, 0] + (torch.rand(B, generator=g, dtype=torch.float64) - 0.5) * 0.8
        old_v[idx] = vl + torch.randn(B, generator=g, dtype=torch.float64) * 0.1
        tgt[idx] = vl + torch.randn(B, generator=g, dtype=torch.float64) * 0.2
        anchor[idx] = (lg + torch.randn(lg.shape, generator=g, dtype=torch.float64) * 0.7).float()
    for k, v in (("old_lp", old_lp), ("old_v", old_v), ("tgt", tgt)):
        t[k] = v.to(torch.float32).to(DEV).contiguous()
    coef, kl_coef = (0.2, 0.01, 0.5, 0.0), 0.7
    total_ref, aux = anchor_kl_ref.loss_fn(lg, vl, mask[idx], action[idx], old_lp[idx], old_v[idx], adv[idx], tgt[idx],
                                           anchor_logits=anchor[idx].double(), anchor_kl_coef=kl_coef, masked_policy=masked,
                                           clip_eps=coef[0], ent_coef=coef[1], vf_coef=coef[2])
    total_ref.backward()
    dzs = [z.grad for z in zs] + [lg.grad, vl.grad[:, None]]
    ins = hs[:4] + [hs[4], hs[4]]
    bound = {}
    for i in range(6):
        bound[f"w{i}"] = (ins[i].detach().abs().T @ dzs[i].abs()).numpy().reshape(-1)
        bound[f"b{i}"] = dzs[i].abs().sum(0).numpy().reshape(-1)
    want = np.array([float(total_ref.detach())] + [float(a.detach()) for a in aux])
    assert want[7] > 0.05  # the KL term is not negligible
    blob = ops.mlp_pack_train(flatten_params(params)[0])
    scratch = torch.full((int(ops._lib.load().brl_mlp_train_scratch_bytes(B)),), 0xFF, dtype=torch.uint8, device=DEV)
    anchor_d = anchor.to(DEV).contiguous()
    first = None
    for call in range(2):  # poisoned scratch, then a second call on the same scratch
        grads, stats, acc = _call(t, blob, B, coef, anchor=anchor_d, kl=kl_coef, scratch=scratch, tune=tune, masked_policy=masked)
        got = stats.cpu().numpy()
        np.testing.assert_allclose(got, want, rtol=5e-5, atol=2e-5, err_msg=f"call {call}")
        gg = grads.cpu().numpy()
        assert np.isfinite(gg).all()
        off = 0
        for k in [f"{c}{i}" for i in range(6) for c in ("w", "b")]:
            want_g = ref[k].grad.numpy().reshape(-1)
            got_g = gg[off:off + want_g.size]
            off += want_g.size
            scale = np.abs(want_g).max()
            tol = 2e-4 * scale + 2e-5 * bound[k]
            bad = np.abs(got_g - want_g) > tol
            assert not bad.any(), (call, k, int(bad.sum()), float(np.abs(got_g - want_g).max()), scale)
        if first is None:
            first = (grads.clone(), stats.clone())
        else:
            assert torch.equal(_bits(first[0]), _bits(grads)) and torch.equal(_bits(first[1]), _bits(stats))


@pytest.mark.parametrize("B,obs_dtype,coef,flags", [
    (1024, torch.bfloat16, (0.2, 0.01, 0.5, 0.0), dict(masked_policy=True, illegal_stat=True)),
    (1000, torch.uint8, (0.1, 0.003, 0.7, 0.3), dict(masked_policy=False, reward_scaling=True)),
])
def test_zero_coefficient_is_bit_equal_to_ppo_grad(B, obs_dtype, coef, flags):
    from brl_b200 import ops
    from brl_b200.optim import flatten_params
    params, t = _learner(61, 3000, B, obs_dtype)
    blob = ops.mlp_pack_train(flatten_params(params)[0])
    g0, s0, a0 = _call(t, blob, B, coef, **flags)
    g1, s1, a1 = _call(t, blob, B, coef, anchor=_anchor_rows(8, 3000), kl=0.0, **flags)
    assert torch.equal(_bits(g0), _bits(g1))
    assert torch.equal(_bits(s0[:7]), _bits(s1[:7]))
    assert float(s0[7]) == 0.0 and float(s1[7]) > 0.0
    assert float(a0[14]) == pytest.approx(float(a1[14]), rel=1e-12)


@pytest.mark.parametrize("K,B,obs_dtype,tune,masked", [
    (1, 1024, torch.bfloat16, 0, True),
    (2, 1000, torch.uint8, 0, False),
    (3, 1024, torch.float32, 4 | 16, True),
    (5, 1000, torch.bfloat16, 16, True),
])
def test_grouped_anchored_equals_solo_anchored_calls(K, B, obs_dtype, tune, masked):
    from brl_b200 import _lib, ops
    from brl_b200.optim import flatten_params
    n, stride, nb = ops.mlp_num_params(), ops.mlp_param_stride(), int(_lib.load().brl_mlp_train_blob_bytes())
    learners = [_learner(71 + k, 2500 + 300 * k, B, obs_dtype) for k in range(K)]
    anchors = [_anchor_rows(90 + k, 2500 + 300 * k) for k in range(K)]  # a different anchor per learner
    kls = [0.5, 0.0, 2.0, 0.1, 1.0][:K]                                   # mixed coefficients, one of them 0
    blob = torch.empty((K, nb), dtype=torch.uint8, device=DEV)
    for k, (params, _) in enumerate(learners):
        ops.mlp_pack_train(flatten_params(params)[0], out=blob[k])
    cfg = dict(masked_policy=masked, value_clipping=True, reward_scaling=False)
    want = [_call(t, blob[k], B, _COEFS[k], anchor=anchors[k], kl=kls[k], tune=tune, **cfg) for k, (_, t) in enumerate(learners)]
    traj = torch.tensor([_row(t) for _, t in learners], dtype=torch.int64, device=DEV)
    coef_t = torch.tensor(_COEFS[:K], dtype=torch.float32, device=DEV)
    table = torch.tensor([a.data_ptr() for a in anchors], dtype=torch.int64, device=DEV)
    kl_t = torch.tensor(kls, dtype=torch.float32, device=DEV)
    scratch = torch.full((ops.ppo_grad_grouped_scratch_bytes(K, B),), 0xFF, dtype=torch.uint8, device=DEV)
    acc = torch.empty((K, _lib.PPO_SCRATCH_BYTES // 8), dtype=torch.float64, device=DEV)
    for call in range(2):
        acc.view(torch.uint8).fill_(0xFF)
        grads = torch.full((K, stride), float("nan"), device=DEV)
        stats = torch.full((K, 8), float("nan"), device=DEV)
        ops.ppo_grad_grouped(traj, coef_t, blob, scratch, grads, stats, acc, batch=B, obs_dtype=obs_dtype, tune=tune,
                             anchor_logits=table, kl_coef=kl_t, **cfg)
        torch.cuda.synchronize()
        for k in range(K):
            g_w, s_w, a_w = want[k]
            assert torch.equal(_bits(grads[k, :n]), _bits(g_w)), (call, k)
            assert torch.equal(_bits(stats[k]), _bits(s_w)), (call, k, stats[k].tolist(), s_w.tolist())
            assert abs(float(acc[k, 14]) - float(a_w[14])) <= 1e-12 * float(a_w[14]), (call, k)
            assert float(stats[k, 7]) > 0.0


@pytest.mark.parametrize("graph", [True, False])
def test_roll_out_records_the_anchor_logits(graph, monkeypatch):
    from brl_b200 import ops, random as brandom
    from brl_b200.deals import synthetic_deal_table
    from brl_b200.env import BridgeBidding
    from brl_b200.models import LAYERS, init_params, make_forward_pass
    from brl_b200.roll_out import make_roll_out
    if not graph:
        monkeypatch.setenv("BRL_ROLLOUT_GRAPH", "0")
    env = BridgeBidding(table=synthetic_deal_table(5000, seed=8), device=DEV)
    n, T = 4096, 4
    config = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode="competitive",
                  num_steps=T, reward_scale=7600.0)
    params, opp, anchor = init_params(101, DEV), init_params(102, DEV), init_params(103, DEV)
    fp = make_forward_pass("relu", "DeepMind")
    roll_out = make_roll_out(config, env, fp, fp, make_forward_pass("relu", "DeepMind"))
    keys = env.make_keys(5, n)
    packed = ops.mlp_pack([anchor[x]["w"] for x in LAYERS], [anchor[x]["b"] for x in LAYERS])
    scratch = ops.mlp_scratch(n, DEV)
    runs = {}
    for anchored in (False, True, True):  # plain, anchored (graph capture on that path), anchored again (replay)
        state = env.init(keys)
        runner = (params, None, state, state.observation, torch.zeros((), dtype=torch.int64, device=DEV), brandom.PRNGKey(9))
        runner, traj = roll_out(runner, opp, anchor_params=anchor if anchored else None)
        torch.cuda.synchronize()
        runs.setdefault(anchored, []).append([getattr(traj, k).clone() for k in traj._fields])
        if not anchored:
            assert roll_out.anchor_logits is None
            continue
        got = roll_out.anchor_logits
        assert got.shape == (T, n, 38) and got.dtype == torch.float32
        for t in range(T):
            want = torch.empty((n, 38), dtype=torch.float32, device=DEV)
            ops.mlp_forward(traj.obs[t].contiguous(), packed, scratch, want, torch.empty(n, device=DEV))
            torch.cuda.synchronize()
            assert torch.equal(_bits(got[t]), _bits(want)), t
    # the anchor changes nothing the trajectory records
    for other in runs[True]:
        assert all(torch.equal(a, b) for a, b in zip(runs[False][0], other))


def _train_config(tmp_path, name, **kw):
    base = dict(num_envs=128, num_steps=4, minibatch_size=128, update_epochs=2, total_timesteps=128 * 4 * 3, hash_size=20,
                num_eval_envs=64, num_prioritized_envs=32, num_eval_step=2, save_model=False, log_path=str(tmp_path), exp_name=name)
    base.update(kw)
    return base


def _save_net(tmp_path, seed, name):
    from brl_b200 import ppo
    from brl_b200.models import init_params
    path = str(tmp_path / f"{name}.pkl")
    ppo.save_params(init_params(seed, DEV), path)
    return path


def _same_runs(a, b, skip=()):
    from brl_b200.models import params_to_numpy
    (runner_a, logs_a), (runner_b, logs_b) = a, b
    assert len(logs_a) == len(logs_b)
    for la, lb in zip(logs_a, logs_b):
        keys = sorted(x for x in lb if not x.startswith("time/") and x not in skip)
        assert keys == sorted(x for x in la if not x.startswith("time/") and x not in skip)
        for x in keys:
            np.testing.assert_allclose(la[x], lb[x], rtol=1e-12, atol=0, err_msg=x)
    pa, pb = params_to_numpy(runner_a[0]), params_to_numpy(runner_b[0])
    assert all((pa[x] == pb[x]).all() for x in pa)


def test_train_with_a_zero_coefficient_anchor_equals_train_without(tmp_path):
    from brl_b200 import ppo, random as brandom
    from brl_b200.deals import synthetic_deal_table
    tables, eval_table = [synthetic_deal_table(300, seed=k) for k in range(2)], synthetic_deal_table(200, seed=9)
    anchor = _save_net(tmp_path, 7, "anchor")
    plain = ppo.train(_train_config(tmp_path, "a", lr=1e-4), brandom.PRNGKey(3), tables=tables, eval_table=eval_table, device=DEV)
    anch = ppo.train(_train_config(tmp_path, "b", lr=1e-4, anchor_model_path=anchor, anchor_kl_coef=0.0), brandom.PRNGKey(3),
                     tables=tables, eval_table=eval_table, device=DEV)
    _same_runs(anch, plain, skip=("train/anchor_kl",))
    assert all("train/anchor_kl" in log and log["train/anchor_kl"] > 0 for log in anch[1])
    assert all("train/anchor_kl" not in log for log in plain[1])


def test_train_population_with_anchors_equals_solo_anchored_runs(tmp_path):
    from brl_b200 import ppo, random as brandom
    from brl_b200.deals import synthetic_deal_table
    tables, eval_table = [synthetic_deal_table(300, seed=k) for k in range(2)], synthetic_deal_table(200, seed=9)
    anchors = [_save_net(tmp_path, 11, "a0"), _save_net(tmp_path, 12, "a1")]

    def configs(tag):
        return [_train_config(tmp_path, f"{tag}0", seed=0, lr=1e-4, anchor_model_path=anchors[0], anchor_kl_coef=0.5),
                _train_config(tmp_path, f"{tag}1", seed=1, lr=3e-4, ent_coef=0.01, anchor_model_path=anchors[1], anchor_kl_coef=2.0)]
    seen = [[], []]
    pop = ppo.train_population(configs("p"), [brandom.PRNGKey(20), brandom.PRNGKey(21)], tables=tables, eval_table=eval_table,
                               device=DEV, log_fns=[s.append for s in seen])
    for k, cfg in enumerate(configs("s")):
        solo = ppo.train(cfg, brandom.PRNGKey(20 + k), tables=tables, eval_table=eval_table, device=DEV)
        assert seen[k] == pop[k][1]
        _same_runs(pop[k], solo)
        assert all(log["train/anchor_kl"] > 0 for log in pop[k][1])


def test_a_large_coefficient_keeps_the_policy_near_its_anchor(tmp_path):
    """anchor = the initial model, a large learning rate: after a few iterations the KL to the anchor is smaller at
    anchor_kl_coef = 10 than at 0"""
    from brl_b200 import ppo, random as brandom
    from brl_b200.deals import synthetic_deal_table
    tables, eval_table = [synthetic_deal_table(300, seed=k) for k in range(2)], synthetic_deal_table(200, seed=9)
    anchor = _save_net(tmp_path, 13, "anchor")
    kl = {}
    for coef in (0.0, 10.0):
        cfg = _train_config(tmp_path, f"c{coef}", lr=1e-3, total_timesteps=128 * 4 * 4, load_initial_model=True,
                            initial_model_path=anchor, anchor_model_path=anchor, anchor_kl_coef=coef)
        _, logs = ppo.train(cfg, brandom.PRNGKey(4), tables=tables, eval_table=eval_table, device=DEV)
        kl[coef] = logs[-1]["train/anchor_kl"]
    assert kl[10.0] < kl[0.0], kl
