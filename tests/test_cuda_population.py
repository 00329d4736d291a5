"""Population training on one GPU: K learners' optimizer steps as one grouped step (brl_ppo_grad_grouped,
brl_mlp_adam_step_grouped, update.make_population_update_step).  Every learner's results must be bit-identical to
its solo call; the solo path itself is checked against float64 in test_cuda_ppo.py."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t.contiguous().view(torch.int64)


def _learner(seed, total, B, obs_dtype):
    """one learner's net, trajectory and minibatch index (the buffers of ops.ppo_grad)"""
    from brl_b200.models import init_params
    g = torch.Generator().manual_seed(seed)
    params = init_params(seed, DEV)
    for name in params:  # non-zero biases: every bias path is exercised
        params[name]["b"] = torch.randn(params[name]["b"].shape, generator=g).to(DEV) * 0.05
    obs = (torch.rand((total, 480), generator=g) < 0.05).to(obs_dtype).to(DEV)
    mask = torch.rand((total, 38), generator=g) < 0.5
    mask[:, 0] = True
    action = torch.multinomial(mask.float(), 1, generator=g)[:, 0].to(torch.int32)
    f32 = lambda t: t.to(torch.float32).to(DEV).contiguous()  # noqa: E731
    traj = dict(obs=obs, mask=mask.to(torch.uint8).to(DEV), action=action.to(DEV),
                old_lp=f32(-torch.rand(total, generator=g) * 3), old_v=f32(torch.randn(total, generator=g) * 0.3),
                adv=f32(torch.randn(total, generator=g)), tgt=f32(torch.randn(total, generator=g) * 0.3),
                index=torch.randperm(total, generator=g)[:B].to(torch.int32).to(DEV))
    return params, traj


def _row(t):
    from brl_b200 import ops
    return ops.ppo_trajectory_row(t["obs"], t["index"], t["mask"], t["action"], t["old_lp"], t["old_v"], t["adv"], t["tgt"])


# per-learner coefficients, all different; learner 1 has a non-zero illegal-action coefficient
_COEFS = [(0.2, 0.01, 0.5, 0.0), (0.1, 0.003, 0.7, 0.3), (0.3, 0.02, 0.25, 0.0), (0.15, 0.0, 1.0, 0.0), (0.25, 0.05, 0.4, 0.0)]


@pytest.mark.parametrize("K,B,obs_dtype,tune,flags,illegal_stat", [
    (1, 1024, torch.bfloat16, 0, (True, False, True), True),
    (2, 1000, torch.uint8, 0, (True, False, True), False),      # ragged B: row / K tails in every learner's GEMMs
    (3, 1024, torch.float32, 4 | 16, (False, True, True), True),  # the other tile widths; reward scaling (prepass)
    (3, 1000, torch.bfloat16, 4, (True, True, False), False),
    (5, 1000, torch.bfloat16, 16, (True, False, True), True),
    (5, 1024, torch.uint8, 0, (False, False, True), False),
])
def test_grouped_gradient_equals_solo_calls(K, B, obs_dtype, tune, flags, illegal_stat):
    from brl_b200 import _lib, ops
    from brl_b200.optim import flatten_params
    value_clipping, reward_scaling, masked = flags
    n, stride, nb = ops.mlp_num_params(), ops.mlp_param_stride(), int(_lib.load().brl_mlp_train_blob_bytes())
    learners = [_learner(11 + k, 2500 + 300 * k, B, obs_dtype) for k in range(K)]  # separate allocations, different sizes
    coefs = _COEFS[:K]
    blob = torch.empty((K, nb), dtype=torch.uint8, device=DEV)
    flat = []
    for k, (params, _) in enumerate(learners):
        fp, _ = flatten_params(params)
        flat.append(fp)
        ops.mlp_pack_train(fp, out=blob[k])
    cfg = dict(value_clipping=value_clipping, reward_scaling=reward_scaling, masked_policy=masked)
    # solo calls
    want = []
    for k, (_, t) in enumerate(learners):
        grads = torch.full((n,), float("nan"), device=DEV)
        stats = torch.zeros(8, device=DEV)
        acc = ops.ppo_scratch(DEV)
        c = coefs[k]
        ops.ppo_grad(t["obs"], blob[k], ops.mlp_train_scratch(B, DEV), t["index"], t["mask"], t["action"], t["old_lp"], t["old_v"],
                     t["adv"], t["tgt"], grads, stats, acc, clip_eps=c[0], ent_coef=c[1], vf_coef=c[2], illegal_l2_coef=c[3],
                     illegal_stat=illegal_stat, tune=tune, **cfg)
        want.append((grads, stats, float(acc[14])))
    # grouped calls: poisoned scratch, two calls back to back on it
    traj = torch.tensor([_row(t) for _, t in learners], dtype=torch.int64, device=DEV)
    coef_t = torch.tensor(coefs, dtype=torch.float32, device=DEV)
    scratch = torch.full((ops.ppo_grad_grouped_scratch_bytes(K, B),), 0xFF, dtype=torch.uint8, device=DEV)
    acc = torch.empty((K, _lib.PPO_SCRATCH_BYTES // 8), dtype=torch.float64, device=DEV)
    for call in range(2):
        acc.view(torch.uint8).fill_(0xFF)
        grads = torch.full((K, stride), float("nan"), device=DEV)
        stats = torch.full((K, 8), float("nan"), device=DEV)
        ops.ppo_grad_grouped(traj, coef_t, blob, scratch, grads, stats, acc, batch=B, obs_dtype=obs_dtype,
                             illegal_stat=illegal_stat, tune=tune, **cfg)
        torch.cuda.synchronize()
        for k in range(K):
            g_w, s_w, ss_w = want[k]
            assert torch.equal(_bits(grads[k, :n]), _bits(g_w)), (call, k)
            assert torch.equal(_bits(stats[k, :7]), _bits(s_w[:7])), (call, k, stats[k].tolist(), s_w.tolist())
            assert abs(float(acc[k, 14]) - ss_w) <= 1e-12 * ss_w, (call, k)
            assert bool(torch.isnan(stats[k, 6])) == (not illegal_stat and coefs[k][3] == 0.0)
        assert bool(torch.isnan(grads[:, n:]).all())  # the rows' padding is not written


def test_grouped_learner_matches_float64_autograd():
    """learner 1 of a K = 3 call against float64 autograd of the restated loss and net (oracle/ppo_ref.py), at the bars
    of test_cuda_ppo.py::test_ppo_grad_matches_float64_autograd"""
    from brl_b200 import _lib, ops
    from brl_b200.models import params_to_numpy
    from brl_b200.optim import flatten_params
    from oracle import ppo_ref
    K, B, total = 3, 1000, 3000
    learners = [_learner(21 + k, total, B, torch.uint8) for k in range(K)]
    params, t = learners[1]
    obs = t["obs"].cpu().bool()
    # rows whose hidden pre-activations stay 2e-5 from zero in float64 (the ReLU kink, as in test_cuda_ppo.py)
    pn = {k: torch.tensor(v, dtype=torch.float64) for k, v in params_to_numpy(params).items()}
    h, margin = obs.double(), torch.full((total,), float("inf"), dtype=torch.float64)
    for i in range(4):
        z = h @ pn[f"w{i}"] + pn[f"b{i}"]
        margin = torch.minimum(margin, z.abs().min(dim=1).values)
        h = torch.relu(z)
    safe = torch.nonzero(margin > 2e-5)[:, 0]
    assert len(safe) >= B
    g = torch.Generator().manual_seed(5)
    idx = safe[torch.randperm(len(safe), generator=g)[:B]]
    t["index"] = idx.to(torch.int32).to(DEV)
    mask, action = t["mask"].cpu().bool(), t["action"].cpu()
    ref = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in params_to_numpy(params).items()}
    hs, zs = [obs[idx].double()], []
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
    with torch.no_grad():  # old log-probs near the current policy: ratios straddle the clip range
        ml = torch.where(mask[idx], lg, torch.tensor(float("-inf"), dtype=torch.float64))
        old_lp[idx] = torch.log_softmax(ml, 1).gather(1, action[idx].long()[:, None])[:, 0] + (torch.rand(B, generator=g, dtype=torch.float64) - 0.5) * 0.8
        old_v[idx] = vl + torch.randn(B, generator=g, dtype=torch.float64) * 0.1
        tgt[idx] = vl + torch.randn(B, generator=g, dtype=torch.float64) * 0.2
    for k, v in (("old_lp", old_lp), ("old_v", old_v), ("tgt", tgt)):
        t[k] = v.to(torch.float32).to(DEV).contiguous()
    c = _COEFS[1][:3]
    total_ref, aux = ppo_ref.loss_fn(lg, vl, mask[idx], action[idx], old_lp[idx], old_v[idx], adv[idx], tgt[idx],
                                     clip_eps=c[0], ent_coef=c[1], vf_coef=c[2])
    total_ref.backward()
    dzs = [z.grad for z in zs] + [lg.grad, vl.grad[:, None]]
    ins = hs[:4] + [hs[4], hs[4]]
    bound = {}
    for i in range(6):
        bound[f"w{i}"] = (ins[i].detach().abs().T @ dzs[i].abs()).numpy().reshape(-1)
        bound[f"b{i}"] = dzs[i].abs().sum(0).numpy().reshape(-1)
    nb = int(_lib.load().brl_mlp_train_blob_bytes())
    blob = torch.empty((K, nb), dtype=torch.uint8, device=DEV)
    for k, (p, _) in enumerate(learners):
        ops.mlp_pack_train(flatten_params(p)[0], out=blob[k])
    coefs = torch.tensor([_COEFS[0], _COEFS[1][:3] + (0.0,), _COEFS[2]], dtype=torch.float32, device=DEV)
    grads = torch.full((K, ops.mlp_param_stride()), float("nan"), device=DEV)
    stats = torch.zeros((K, 8), device=DEV)
    acc = torch.zeros((K, _lib.PPO_SCRATCH_BYTES // 8), dtype=torch.float64, device=DEV)
    scratch = torch.full((ops.ppo_grad_grouped_scratch_bytes(K, B),), 0xFF, dtype=torch.uint8, device=DEV)
    traj = torch.tensor([_row(tt) for _, tt in learners], dtype=torch.int64, device=DEV)
    ops.ppo_grad_grouped(traj, coefs, blob, scratch, grads, stats, acc, batch=B, obs_dtype=torch.uint8)
    got = stats[1].cpu().numpy()
    want = np.array([float(total_ref.detach())] + [float(a.detach()) for a in aux])
    np.testing.assert_allclose(got[:7], want, rtol=5e-5, atol=5e-6)
    gg = grads[1, :ops.mlp_num_params()].cpu().numpy()
    assert np.isfinite(gg).all()
    np.testing.assert_allclose(float(acc[1, 14]), float((gg.astype(np.float64) ** 2).sum()), rtol=1e-5)
    off = 0
    for k in [f"{c}{i}" for i in range(6) for c in ("w", "b")]:
        want_g = ref[k].grad.numpy().reshape(-1)
        got_g = gg[off:off + want_g.size]
        off += want_g.size
        scale = np.abs(want_g).max()
        tol = 2e-4 * scale + 2e-5 * bound[k]
        bad = np.abs(got_g - want_g) > tol
        assert not bad.any(), (k, int(bad.sum()), float(np.abs(got_g - want_g).max()), scale)
    assert off == gg.size


def test_grouped_adam_equals_solo_steps():
    """params, m, v and the blob rows after brl_mlp_adam_step_grouped equal K solo brl_mlp_adam_step calls, with a
    different step count, learning rate and clipping per learner"""
    from brl_b200 import _lib, ops
    K = 4
    n, stride, nb = ops.mlp_num_params(), ops.mlp_param_stride(), int(_lib.load().brl_mlp_train_blob_bytes())
    g = torch.Generator(device=DEV).manual_seed(1)
    p = torch.randn((K, stride), device=DEV, generator=g) * 0.05
    grads = torch.randn((K, stride), device=DEV, generator=g) * torch.tensor([1.0, 1e-3, 0.3, 3.0], device=DEV)[:, None]
    m = torch.randn((K, stride), device=DEV, generator=g) * 1e-3
    v = torch.rand((K, stride), device=DEV, generator=g) * 1e-5
    acc = torch.zeros((K, _lib.PPO_SCRATCH_BYTES // 8), dtype=torch.float64, device=DEV)
    acc[:, 14] = (grads[:, :n].double() ** 2).sum(1)
    blob = torch.empty((K, nb), dtype=torch.uint8, device=DEV)
    for k in range(K):
        ops.mlp_pack_train(p[k, :n].contiguous(), out=blob[k])
    steps, lrs, clips = [1, 7, 100, 3], [1e-3, 3e-4, 2e-3, 5e-5], [0.5, 0.0, 10.0, 0.5]
    solo = [(p[k, :n].clone(), m[k, :n].clone(), v[k, :n].clone(), blob[k].clone()) for k in range(K)]
    for k, (sp, sm, sv, sb) in enumerate(solo):
        ops.mlp_adam_step(sp, grads[k, :n].contiguous(), sm, sv, acc[k, 14:15].contiguous(), sb, step=steps[k], lr=lrs[k],
                          max_grad_norm=clips[k])
    ops.mlp_adam_step_grouped(p, grads, m, v, acc, blob, steps=steps, lrs=lrs, max_grad_norms=clips)
    torch.cuda.synchronize()
    for k, (sp, sm, sv, sb) in enumerate(solo):
        assert torch.equal(_bits(p[k, :n]), _bits(sp)), k
        assert torch.equal(_bits(m[k, :n]), _bits(sm)), k
        assert torch.equal(_bits(v[k, :n]), _bits(sv)), k
        assert torch.equal(blob[k], sb), k
    # no learners: a no-op that reads nothing
    e = torch.empty((0, stride), device=DEV)
    ops.mlp_adam_step_grouped(e, e, e, e, torch.empty((0, _lib.PPO_SCRATCH_BYTES // 8), dtype=torch.float64, device=DEV),
                              torch.empty((0, nb), dtype=torch.uint8, device=DEV), steps=[], lrs=[], max_grad_norms=[])


def _rollout(seed, T, n):
    from brl_b200.roll_out import Transition
    g = torch.Generator().manual_seed(seed)
    obs = (torch.rand((T, n, 480), generator=g) < 0.04).to(torch.bfloat16)
    mask = torch.rand((T, n, 38), generator=g) < 0.5
    mask[..., 0] = True
    action = torch.multinomial(mask.reshape(-1, 38).float(), 1, generator=g)[:, 0].to(torch.int32).reshape(T, n)
    traj = Transition(done=torch.zeros((T, n), dtype=torch.bool, device=DEV), action=action.to(DEV),
                      value=(torch.randn((T, n), generator=g) * 0.3).to(DEV), reward=torch.zeros((T, n), device=DEV),
                      log_prob=(-torch.rand((T, n), generator=g) * 3).to(DEV), obs=obs.to(DEV), legal_action_mask=mask.to(DEV))
    return traj, torch.randn((T, n), generator=g).to(DEV), (torch.randn((T, n), generator=g) * 0.3).to(DEV)


@pytest.mark.parametrize("stat_mode", ["last", "all"])
def test_population_update_step_equals_solo_update_steps(stat_mode):
    from brl_b200 import random as brandom
    from brl_b200.models import init_params, make_forward_pass, params_to_numpy
    from brl_b200.optim import make_optimizer
    from brl_b200.update import make_population_update_step, make_update_step
    T, n, mbs, epochs = 8, 256, 512, 3
    nmb = T * n // mbs
    base = dict(actor_illegal_action_mask=True, clip_eps=0.2, ent_coef=0.001, vf_coef=0.5, illegal_action_l2norm_coef=0.0,
                value_clipping=True, reward_scaling=False, num_minibatches=nmb, minibatch_size=mbs, update_epochs=epochs,
                num_steps=T, num_envs=n, total_timesteps=T * n * 4, num_updates=4, lr=1e-3, anneal_lr=False, max_grad_norm=0.5,
                global_gradient_clipping=True, illegal_action_loss_stat=stat_mode, actor_model_type="DeepMind",
                actor_activation="relu")
    configs = [dict(base), dict(base, lr=3e-4, ent_coef=0.01, clip_eps=0.1, anneal_lr=True),
               dict(base, lr=2e-3, vf_coef=0.8, max_grad_norm=0.2, illegal_action_l2norm_coef=0.2)]
    fp = make_forward_pass("relu", "DeepMind", precision="tc")

    def perm(rng, bs):
        return torch.randperm(bs, generator=torch.Generator().manual_seed(rng & 0x7FFFFFFF))

    rollouts = [_rollout(40 + k, T, n) for k in range(3)]
    runners = []
    for k in range(3):
        params = init_params(30 + k, DEV)
        runners.append((params, None, None, None, 0, brandom.PRNGKey(k)))
    solo = []
    for k, c in enumerate(configs):
        opt = make_optimizer(c)
        step = make_update_step(c, fp, opt, permutation_fn=perm)
        rs = runners[k]
        rs = (rs[0], opt.init(rs[0])) + rs[2:]
        out = step(rs, *rollouts[k])
        out = step(out[0], *rollouts[k])  # a second update: counts > 0, annealed lr
        solo.append(out)
    opts = [make_optimizer(c) for c in configs]
    pop = make_population_update_step(configs, fp, opts, permutation_fn=perm)
    rs = [(r[0], o.init(r[0])) + r[2:] for r, o in zip(runners, opts)]
    outs = pop(rs, [r[0] for r in rollouts], [r[1] for r in rollouts], [r[2] for r in rollouts])
    outs = pop([o[0] for o in outs], [r[0] for r in rollouts], [r[1] for r in rollouts], [r[2] for r in rollouts])
    for k in range(3):
        (p_s, st_s, *_, rng_s), (tl_s, aux_s) = solo[k]
        (p_g, st_g, *_, rng_g), (tl_g, aux_g) = outs[k]
        assert rng_s == rng_g and st_s.count == st_g.count == 2 * epochs * nmb
        for name, w in params_to_numpy(p_s).items():
            assert np.array_equal(w, params_to_numpy(p_g)[name]), (k, name)
        assert torch.equal(_bits(st_s.mu), _bits(st_g.mu)) and torch.equal(_bits(st_s.nu), _bits(st_g.nu)), k
        for a, b in zip((tl_s,) + tuple(aux_s), (tl_g,) + tuple(aux_g)):
            assert torch.equal(_bits(a), _bits(b)), k  # NaN (statistic not formed) in the same places
        if stat_mode == "last":
            assert bool(torch.isnan(aux_s[5][:, 0]).all()) == (configs[k]["illegal_action_l2norm_coef"] == 0.0)


def _population_configs(tmp_path):
    base = dict(num_envs=128, num_steps=4, minibatch_size=128, update_epochs=2, total_timesteps=128 * 4 * 3, hash_size=20,
                num_eval_envs=64, num_prioritized_envs=32, num_eval_step=2, save_model=True, log_path=str(tmp_path))
    return [dict(base, seed=0, lr=1e-4, ent_coef=0.001, exp_name="a", ratio_model_zoo=1.0, prioritized_fictitious=True),  # PFSP
            dict(base, seed=1, lr=3e-4, ent_coef=0.01, exp_name="b", ratio_model_zoo=0.5),                               # FSP
            dict(base, seed=2, lr=2e-5, ent_coef=0.0, exp_name="c", anneal_lr=True, clip_eps=0.1)]                       # self-play


@pytest.mark.parametrize("K", [1, 3])
def test_train_population_equals_solo_train_runs(K, tmp_path, monkeypatch):
    """each learner of train_population has the logs (every key but time/*) and final parameters of ppo.train with its
    config and rng; learner 0 runs PFSP on a device zoo, and the tables rotate"""
    from brl_b200 import ppo, random as brandom
    from brl_b200.deals import synthetic_deal_table
    from brl_b200.models import params_to_numpy
    made = []

    class RecordedZoo(ppo.ModelZoo):
        def __init__(self, *a):
            super().__init__(*a)
            made.append(self)
    monkeypatch.setattr(ppo, "ModelZoo", RecordedZoo)
    tables = [synthetic_deal_table(300, seed=k) for k in range(3)]
    eval_table = synthetic_deal_table(200, seed=9)
    configs = _population_configs(tmp_path / "pop")[:K]
    seen = [[] for _ in range(K)]
    pop = ppo.train_population(configs, [brandom.PRNGKey(10 + k) for k in range(K)], tables=tables, eval_table=eval_table,
                               device=DEV, log_fns=[s.append for s in seen])
    assert len(made) == (1 if K == 1 else 2)  # one device zoo per learner with ratio_model_zoo > 0
    solo_configs = _population_configs(tmp_path / "solo")[:K]
    for k in range(K):
        solo = ppo.train(solo_configs[k], brandom.PRNGKey(10 + k), tables=tables, eval_table=eval_table, device=DEV)
        (runner_p, logs_p), (runner_s, logs_s) = pop[k], solo
        assert seen[k] == logs_p and len(logs_p) == len(logs_s) == 3
        for lp, ls in zip(logs_p, logs_s):
            keys = sorted(x for x in ls if not x.startswith("time/"))
            assert keys == sorted(x for x in lp if not x.startswith("time/"))
            for x in keys:
                np.testing.assert_allclose(lp[x], ls[x], rtol=1e-12, atol=0, err_msg=f"learner {k}: {x}")
        assert any("table" in log for log in logs_p), "hash_size=20 boards must trigger a table rotation"
        pp, ps = params_to_numpy(runner_p[0]), params_to_numpy(runner_s[0])
        assert all((pp[x] == ps[x]).all() for x in pp), k
        assert runner_p[1].count == runner_s[1].count == 3 * 2 * 4
