"""GPU: call-value policy improvement (DESIGN.md f17).  brl_cv_grad / brl_cv_eval against float64 autograd of
tests/cvi_ref.py at the bars of test_cuda_sl.py; brl_call_values' training examples against the host loop of
tests/call_values_ref.py bit for bit; the evaluator's examples across chunkings; and cvi.train."""
import os

import numpy as np
import pytest
import torch

from tests import call_values_ref as CR
from tests import cvi_ref as R
from tests import helpers as H
from tests.test_cuda_call_values import FORCE_FUSED, FORCE_LAYERS, _env
from tests.test_cuda_sl import _grad_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _gains(B, seed):
    """gains like brl_call_values': integers in [-12, 12], NaN on illegal calls, at least one legal call per sample"""
    rng = np.random.default_rng(seed)
    g = rng.integers(-12, 13, (B, 38)).astype(np.float32)
    legal = rng.random((B, 38)) < 0.4
    legal[:, 0] = True
    return np.where(legal, g, np.float32("nan"))


def _autograd(params, obs, gain, ent):
    from brl_b200.models import params_to_numpy
    ref = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in params_to_numpy(params).items()}
    hs, zs = [obs.double()], []
    for i in range(4):
        z = hs[-1] @ ref[f"w{i}"] + ref[f"b{i}"]
        z.retain_grad()
        zs.append(z)
        hs.append(torch.relu(z))
    lg = hs[-1] @ ref["w4"] + ref["b4"]
    vl = (hs[-1] @ ref["w5"] + ref["b5"])[:, 0]
    lg.retain_grad()
    total = R.torch_loss(lg, torch.tensor(gain, dtype=torch.float64), ent)
    (total + 0.0 * vl.sum()).backward()
    _, _, stats = R.loss_grad_stats(lg.detach().numpy(), gain, ent)
    dzs = [z.grad for z in zs] + [lg.grad]
    bound = {}
    for i in range(5):
        bound[f"w{i}"] = (hs[i].detach().abs().T @ dzs[i].abs()).numpy().reshape(-1)
        bound[f"b{i}"] = dzs[i].abs().sum(0).numpy().reshape(-1)
    return ref, stats, bound


CASES = [(1, torch.float32, 0.0, 0), (1, torch.uint8, 0.01, 0), (1000, torch.bfloat16, 0.0, 0), (1000, torch.uint8, 0.01, 0),
         (1024, torch.float32, 0.01, 0), (1024, torch.bfloat16, 0.0, 1 << 16 | 1 << 17), (8205, torch.bfloat16, 0.01, 0),
         (8205, torch.uint8, 0.0, 1 << 16 | 1 << 17)]


@pytest.mark.parametrize("B,obs_dtype,ent,tiles", CASES)
def test_cv_grad_matches_float64_autograd(B, obs_dtype, ent, tiles):
    from brl_b200 import ops
    from brl_b200.optim import flatten_params
    params, obs, _, _ = _grad_case(B, 60 + B)
    gain = _gains(B, B)
    ref, want_stats, bound = _autograd(params, obs, gain, ent)
    flat_p, _ = flatten_params(params)
    blob = ops.mlp_pack_train(flat_p)
    scratch = torch.full((ops._lib.load().brl_mlp_train_scratch_bytes(B),), 0xFF, dtype=torch.uint8, device=DEV)  # poisoned
    grads = torch.full_like(flat_p, float("nan"))
    stats = torch.full((8,), float("nan"), device=DEV)
    acc = torch.full((16,), float("nan"), dtype=torch.float64, device=DEV)
    dobs, dgain = obs.to(obs_dtype).to(DEV), torch.as_tensor(gain, device=DEV)
    ops.cv_grad(dobs, blob, scratch, dgain, grads, stats, acc, ent_coef=ent, tiles=tiles)
    got = stats.cpu().numpy()
    np.testing.assert_allclose(got[:7], want_stats[:7], rtol=5e-5, atol=2e-5)
    assert got[7] == 0
    gg = grads.cpu().numpy()
    assert np.isfinite(gg).all()
    np.testing.assert_allclose(float(acc[14]), float((gg.astype(np.float64) ** 2).sum()), rtol=1e-5)
    off = 0
    for k in [f"{c}{i}" for i in range(6) for c in ("w", "b")]:
        n = ref[k].numel()
        got_g = gg[off:off + n]
        off += n
        if k in ("w5", "b5"):
            assert (got_g == 0).all(), k                    # the value head gets no gradient
            continue
        want_g = ref[k].grad.numpy().reshape(-1)
        scale = np.abs(want_g).max()
        tol = 2e-4 * scale + 2e-5 * bound[k]
        bad = np.abs(got_g - want_g) > tol
        assert not bad.any(), (k, int(bad.sum()), float(np.abs(got_g - want_g).max()), scale)
    # a second call on the same scratch, and brl_cv_eval: bit-equal stats, the gradient untouched by eval
    stats2, grads2 = torch.zeros(8, device=DEV), torch.zeros_like(grads)
    ops.cv_grad(dobs, blob, scratch, dgain, grads2, stats2, acc, ent_coef=ent, tiles=tiles)
    assert torch.equal(stats2, stats) and torch.equal(grads2, grads)
    stats_e = torch.zeros(8, device=DEV)
    ops.cv_eval(dobs, blob, scratch, dgain, stats_e, ops.sl_acc(DEV), ent_coef=ent, tiles=tiles)
    assert torch.equal(stats_e, stats) and torch.equal(grads2, grads)


def test_empty_batch_is_a_no_op_and_buffers_are_checked():
    from brl_b200 import _lib, ops
    p = _lib.BrlSlParams(0, 0.0, 0)
    for name, n in (("brl_cv_grad", 7), ("brl_cv_eval", 6)):
        _lib.call(name, torch.cuda.current_stream().cuda_stream, [None] * n, p)
    with pytest.raises(_lib.BrlError, match="NULL"):
        _lib.call("brl_cv_grad", torch.cuda.current_stream().cuda_stream, [None] * 7, _lib.BrlSlParams(4, 0.0, 0))


# ---- brl_call_values' training examples ----------------------------------------------------------------------------
class _Pair:
    """one brl_call_values call with records and one with records + examples, on the same base match"""

    def __init__(self, env, n, nets, models, tune=0, single=False, capacity=None):
        from brl_b200 import ops, random as brandom
        from brl_b200.evaluation import _MatchBuffers
        from brl_b200.models import make_forward_pass
        M, width = len(nets), len(models)
        b = _MatchBuffers(n, M, 0, DEV, with_models=True, with_tables=True, players=width == 4)
        fp = make_forward_pass("relu", "DeepMind", precision="tc-bf16" if single else None)
        size = ops._lib.load().brl_mlp_packed_bytes()
        for m, p in enumerate(nets):
            fp.pack_into(p, b.pool[m, :size])
        _, sub = brandom.split(brandom.PRNGKey(n))
        b.keys.copy_(env.make_keys(sub, n))
        b.env_models.copy_(torch.tensor(models, dtype=torch.int32, device=DEV).expand(n, width))
        b.play(env, single, tune)
        self.match, cap = b, capacity if capacity is not None else 48 * n
        self.out = []
        for train in (False, True):
            o = dict(gain=torch.full((M,) + ops.CALL_GAIN_SHAPE, -1, dtype=torch.int64, device=DEV),
                     regret=torch.full((M,) + ops.CALL_REGRET_SHAPE, -1, dtype=torch.int64, device=DEV),
                     mismatch=torch.full((M,), -1, dtype=torch.int64, device=DEV),
                     status=torch.full((1,), -1, dtype=torch.int32, device=DEV),
                     records=ops.CallValueRecords(cap, DEV, train))
            if train:
                o["records"].obs.fill_(float("nan"))
                o["records"].gain.fill_(-7.0)
            scratch = torch.full((ops.call_values_scratch_bytes(n, M),), 0xFF, dtype=torch.uint8, device=DEV)
            ops.call_values(b.keys, env.table, b.pool, b.env_models, b.tables[0].rewards, b.tables[1].rewards, scratch,
                            o["gain"], o["regret"], o["mismatch"], o["status"], records=o["records"], single_bf16=single,
                            tune=tune)
            self.out.append(o)
        torch.cuda.synchronize()


EX_CASES = [("tc", FORCE_LAYERS, (0, 1)), ("tc-bf16", FORCE_FUSED, (0, 1)), ("tc", FORCE_FUSED, (0, 1, 2, 3)),
            ("tc-bf16", FORCE_LAYERS, (2, 0, 1, 1))]


@pytest.mark.parametrize("precision, tune, models", EX_CASES)
@pytest.mark.parametrize("n", [1, 7, 100, 1000])
def test_examples_equal_the_host_loop(n, precision, tune, models):
    from brl_b200 import ops, random as brandom
    if n == 1000 and (precision, tune, models) != EX_CASES[0]:
        pytest.skip("the 1,000-board host replay runs for one case")
    env = _env()
    M = max(models) + 1
    nets = [H.seeded_params(750 + k, DEV) for k in range(M)]
    run = _Pair(env, n, nets, models, tune, precision == "tc-bf16")
    plain, train = run.out
    for f in ("gain", "regret", "mismatch", "status"):
        assert torch.equal(plain[f], train[f]), f
    assert int(train["status"][0]) == 0
    rp, rt = plain["records"], train["records"]
    k = int(rt.count[0])
    assert int(rp.count[0]) == k
    # the same records: slots follow the gains kernel's atomics, so compare per (env, table) in play order (rising slots)
    cols = ops.CALL_RECORD_FIELDS + ("r",)
    hp, ht = ({f: getattr(r, f)[:k].cpu().numpy() for f in cols} for r in (rp, rt))
    hp["r"], ht["r"] = hp["r"].view(np.uint32), ht["r"].view(np.uint32)
    sp, st = (np.lexsort((h["table"], h["env"])) for h in (hp, ht))
    for f in cols:
        assert np.array_equal(hp[f][sp], ht[f][st]), f
    assert torch.isnan(rt.obs[k:].float()).all() and (rt.gain[k:] == -7.0).all()          # slots beyond the count untouched
    obs = rt.obs[:k].view(torch.int16).cpu().numpy().view(np.uint16)
    gain = rt.gain[:k].cpu().numpy()
    rec = {f: getattr(rt, f)[:k].cpu().numpy() for f in ops.CALL_RECORD_FIELDS + ("r",)}
    ref, R_a, R_b = R.host_records_with_obs(env, nets, models, n, brandom.PRNGKey(n), precision, tune)
    dk, rk = {}, {}
    for idx in range(k):
        dk.setdefault((int(rec["env"][idx]), int(rec["table"][idx])), []).append(idx)
    for idx in range(len(ref["env"])):
        rk.setdefault((int(ref["env"][idx]), int(ref["table"][idx])), []).append(idx)
    assert dk.keys() == rk.keys()
    for key, want in rk.items():
        got = sorted(dk[key])
        assert len(got) == len(want), key
        for a, b in zip(got, want):
            assert np.array_equal(obs[a], ref["obs"][b]), key                               # the forward's input, bit for bit
            g = CR.gains(rec["r"][a], float(R_a[key[0]]), float(R_b[key[0]]), key[1], int(rec["player"][a]))
            legal = np.array([x is not None for x in g])
            assert np.array_equal(np.isnan(gain[a]), ~legal), key
            assert np.array_equal(gain[a][legal], np.array([x for x in g if x is not None], np.float32)), key


def test_examples_capacity_overflow_empty_batch_and_buffer_errors():
    from brl_b200 import _lib, ops
    env = _env()
    nets = [H.seeded_params(760 + k, DEV) for k in range(2)]
    full = _Pair(env, 100, nets, (0, 1), FORCE_FUSED)
    small = _Pair(env, 100, nets, (0, 1), FORCE_FUSED, capacity=10)
    st = small.out[1]
    assert int(st["status"][0]) == ops._lib.MATCH_RECORD_CAPACITY
    for f in ("gain", "regret", "mismatch"):
        assert torch.equal(st[f], full.out[1][f]), f
    # the first 10 slots are decisions of the first base iteration (one per env, table A); the full run's record of that
    # decision is its env's first (an env's slots rise in play order)
    fr, sr = full.out[1]["records"], st["records"]
    pos = {}
    for i in range(int(fr.count[0])):
        pos.setdefault(int(fr.env[i]), i)
    for i in range(10):
        assert int(sr.table[i]) == 0
        j = pos[int(sr.env[i])]
        assert torch.equal(sr.obs[i].view(torch.int16), fr.obs[j].view(torch.int16))
        assert torch.equal(sr.gain[i].view(torch.int32), fr.gain[j].view(torch.int32))
    b = full.match
    e = torch.zeros(0, dtype=torch.int64, device=DEV)
    rec = ops.CallValueRecords(4, DEV, True)
    g0 = full.out[1]["gain"].clone()
    ops.call_values(e, env.table, b.pool, torch.zeros((0, 2), dtype=torch.int32, device=DEV), torch.zeros((0, 4), device=DEV),
                    torch.zeros((0, 4), device=DEV), torch.empty(16, dtype=torch.uint8, device=DEV), full.out[1]["gain"],
                    full.out[1]["regret"], full.out[1]["mismatch"], full.out[1]["status"], records=rec)   # a no-op
    torch.cuda.synchronize()
    assert torch.equal(full.out[1]["gain"], g0)
    scratch = torch.empty(ops.call_values_scratch_bytes(10, 2), dtype=torch.uint8, device=DEV)
    o = full.out[1]
    base = [ops._ptr(x) for x in (b.keys[:10], env.table, b.pool, b.env_models[:10], b.tables[0].rewards[:10],
                                  b.tables[1].rewards[:10], scratch, o["gain"], o["regret"], o["mismatch"], o["status"])]
    p = ops._params(10, k_steps=2, n_deals=env.table.shape[0], seed=4)
    recs = rec.ptrs()
    for bad in (recs[:9] + [None], recs[:8] + [None, recs[9]],              # one of the two
                [None] * 8 + recs[8:],                                      # without the records
                recs[:8] + [recs[8] + 2, recs[9]]):                         # a misaligned obs
        with pytest.raises(_lib.BrlError):
            _lib.call("brl_call_values", torch.cuda.current_stream().cuda_stream, base + bad, p)


def test_evaluator_examples_are_independent_of_chunks():
    from brl_b200 import random as brandom
    from brl_b200.evaluation import make_call_values_evaluate
    env = _env()
    n, M = 60, 2
    nets = [H.seeded_params(770 + k, DEV) for k in range(M)]
    one = make_call_values_evaluate(env, "relu", "DeepMind", n, tune=FORCE_FUSED)(nets, brandom.PRNGKey(5), 1, "train")
    many = make_call_values_evaluate(env, "relu", "DeepMind", n, max_envs=38 * 25,
                                     tune=FORCE_FUSED)(nets, brandom.PRNGKey(5), 1, "train")
    for f in ("gain_sums", "regret_sums", "mismatch"):
        assert (one[f] == many[f]).all(), f

    def rows(out):
        r, ex = out["records"], out["examples"]
        assert ex["obs"].is_cuda and ex["gain"].is_cuda and ex["net"].is_cuda
        assert np.array_equal(ex["net"].cpu().numpy(), r["net"])
        order = np.lexsort((r["table"], r["env"]))  # stable: an (env, table)'s records keep their play order
        return (ex["obs"].view(torch.int16).cpu().numpy()[order], ex["gain"].cpu().numpy().view(np.int32)[order])

    a, b = rows(one), rows(many)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    # matches=[(0, 1)]: only the first of the two matches
    first = make_call_values_evaluate(env, "relu", "DeepMind", n, tune=FORCE_FUSED)(nets, brandom.PRNGKey(5), records="train",
                                                                                    matches=[(0, 1)])
    assert (first["gain_sums"][0] == one["gain_sums"][0]).all()                # net 0 decides in match 0 only
    env = one["records"]["env"]
    assert first["records"]["env"].max() < n and len(first["records"]["env"]) == int((env < n).sum())


# ---- cvi.train -----------------------------------------------------------------------------------------------------------
def _cfg(tmp_path, **kw):
    cfg = dict(boards_per_iter=200, num_iters=2, epochs=2, minibatch_size=256, seed=3, num_eval_envs=100, num_eval_step=1,
               save_model=True, save_model_interval=1, log_path=str(tmp_path), exp_name="run", lr=1e-4, ent_coef=0.01,
               max_grad_norm=0.0)
    cfg.update(kw)
    return cfg


def _table():
    from brl_b200.deals import synthetic_deal_table
    return synthetic_deal_table(5000, seed=4)


def test_train_is_deterministic_saves_and_loads(tmp_path):
    """two runs with one seed: bit-equal parameters and logs (time/* aside).  Gradient clipping is off here: it scales by
    |g|^2, an f64 atomic sum whose last bits may depend on the order of the blocks."""
    from brl_b200 import cvi, ppo
    from brl_b200.models import load_params
    runs = []
    for k in range(2):
        runs.append(cvi.train(_cfg(tmp_path, exp_name=f"run{k}"), 0, _table(), device=DEV))
    (p0, l0), (p1, l1) = runs
    for name in p0:
        for kk in ("w", "b"):
            assert torch.equal(p0[name][kk], p1[name][kk])
    assert len(l0) == 2
    for a, b in zip(l0, l1):
        assert {k for k in a if not k.startswith("time/")} == {k for k in b if not k.startswith("time/")}
        for key in a:
            if not key.startswith("time/"):
                assert a[key] == b[key], key
        assert a["cv/decisions"] > 256 and np.isfinite(a["cv/total_loss"]) and "eval/imp" in a
    assert sorted(os.listdir(tmp_path / "run0")) == ["params-00000001.pkl", "params-00000002.pkl"]
    loaded = load_params(str(tmp_path / "run0" / "params-00000002.pkl"), DEV)
    for name in p0:
        for kk in ("w", "b"):
            assert torch.equal(loaded[name][kk], p0[name][kk])
    # ppo.train starts from it (one tiny iteration), and cvi.train starts from it
    cfg = dict(num_envs=64, num_steps=4, total_timesteps=256, minibatch_size=64, update_epochs=1, num_eval_envs=16,
               num_prioritized_envs=16, save_model=False, hash_size=1000, load_initial_model=True,
               initial_model_path=str(tmp_path / "run0" / "params-00000002.pkl"), log_path=str(tmp_path / "ppo"))
    state, logs = ppo.train(cfg, 0, device=DEV)
    assert len(logs) == 1
    again, _ = cvi.train(_cfg(tmp_path, exp_name="run2", num_iters=1, lr=0.0,
                              initial_model_path=str(tmp_path / "run0" / "params-00000002.pkl")), 0, _table(), device=DEV)
    for name in p0:
        for kk in ("w", "b"):
            assert torch.equal(again[name][kk], p0[name][kk])            # lr = 0 leaves the parameters unchanged


def test_update_loop_matches_a_float64_reference_loop():
    """the Updater on a fixed set of examples against the same minibatches in float64 (Adam eps 1e-5, no clipping), at the
    end-to-end bar of test_cuda_sl.py's sl.train check"""
    from brl_b200 import cvi
    from brl_b200.models import params_to_numpy
    from oracle import sl_ref
    B, mb, epochs, lr, ent = 1024, 256, 2, 1e-4, 0.01
    params, obs, _, _ = _grad_case(B, 91)
    gain = _gains(B, 92)
    cfg = dict(cvi.default_config(), minibatch_size=mb, epochs=epochs, lr=lr, ent_coef=ent, max_grad_norm=0.0)
    upd = cvi.Updater(cfg, params, DEV)
    stats = upd.run(obs.to(torch.bfloat16).to(DEV), torch.as_tensor(gain, device=DEV), cvi.permutation_generator(7, 0))
    assert tuple(stats.shape) == (epochs, B // mb, 8)
    order = [f"{c}{i}" for i in range(6) for c in ("w", "b")]
    ref = {k: torch.tensor(v, dtype=torch.float64) for k, v in params_to_numpy(params).items()}
    p = np.concatenate([ref[k].numpy().reshape(-1) for k in order])
    m, v = np.zeros_like(p), np.zeros_like(p)
    gen = cvi.permutation_generator(7, 0)
    step = 0
    shapes = [(k, ref[k].shape) for k in order]
    for _ in range(epochs):
        perm = torch.randperm(B, generator=gen).numpy()
        for k in range(B // mb):
            idx = perm[k * mb:(k + 1) * mb]
            off, cur = 0, {}
            for name, shp in shapes:
                n = int(np.prod(shp))
                cur[name] = torch.tensor(p[off:off + n].reshape(shp), requires_grad=True)
                off += n
            h = obs[idx].double()
            for i in range(4):
                h = torch.relu(h @ cur[f"w{i}"] + cur[f"b{i}"])
            lg = h @ cur["w4"] + cur["b4"]
            vl = (h @ cur["w5"] + cur["b5"])[:, 0]
            (R.torch_loss(lg, torch.tensor(gain[idx], dtype=torch.float64), ent) + 0.0 * vl.sum()).backward()
            g = np.concatenate([cur[name].grad.numpy().reshape(-1) for name in order])
            p, m, v = sl_ref.adam_step(p, g, m, v, step, lr=lr, eps=1e-5)
            step += 1
    got = upd.flat.cpu().numpy().astype(np.float64)
    p0 = np.concatenate([ref[k].numpy().reshape(-1) for k in order])
    err = np.abs((got - p0) - (p - p0))
    assert np.median(err) <= 0.01 * lr * step, float(np.median(err))          # test_cuda_sl.py's sl.train bars
    assert np.quantile(err, 0.99) <= 0.15 * lr * step, [float(np.quantile(err, q)) for q in (0.5, 0.9, 0.99, 0.999, 1.0)]
    assert np.abs(p - p0).max() > 0.5 * lr


def test_large_lr_on_a_fixed_batch_raises_the_mean_gain():
    from brl_b200 import cvi
    B = 1024
    params, obs, _, _ = _grad_case(B, 93)
    gain = _gains(B, 94)
    cfg = dict(cvi.default_config(), minibatch_size=B, epochs=30, lr=1e-3, ent_coef=0.0, max_grad_norm=0.0)
    upd = cvi.Updater(cfg, params, DEV)
    stats = upd.run(obs.to(torch.bfloat16).to(DEV), torch.as_tensor(gain, device=DEV), cvi.permutation_generator(0, 0))
    s = stats.cpu().numpy()
    assert s[-1, 0, 1] > s[0, 0, 1] + 1.0, (s[0, 0, 1], s[-1, 0, 1])     # mean gbar, IMPs
    assert s[-1, 0, 0] < s[0, 0, 0]


def test_with_an_opponent_only_the_learners_decisions_are_trained_on(tmp_path, monkeypatch):
    from brl_b200 import cvi, ppo
    opp = tmp_path / "opp.pkl"
    ppo.save_params(H.seeded_params(780, DEV), str(opp))
    seen = []
    orig = cvi.Updater.run

    def spy(self, obs, gain, gen):
        seen.append((obs.shape[0], gain.clone()))
        return orig(self, obs, gain, gen)
    monkeypatch.setattr(cvi.Updater, "run", spy)
    calls = []
    from brl_b200 import evaluation
    make = evaluation.make_call_values_evaluate

    def wrap(*a, **k):
        f = make(*a, **k)

        def g(*aa, **kk):
            out = f(*aa, **kk)
            calls.append(out)
            return out
        return g
    monkeypatch.setattr(cvi, "make_call_values_evaluate", wrap)
    _, logs = cvi.train(_cfg(tmp_path, num_iters=1, opponent_model_path=str(opp)), 0, _table(), device=DEV)
    out = calls[0]
    net = out["examples"]["net"].cpu().numpy()
    assert (net == 0).any() and (net == 1).any()
    assert seen[0][0] == int((net == 0).sum()) == logs[0]["cv/decisions"]
    assert torch.equal(seen[0][1].view(torch.int32), out["examples"]["gain"][out["examples"]["net"] == 0].view(torch.int32))
    assert out["records"]["env"].max() < 200                                  # one match: the opponent's self-play is not played
