"""GPU: partnerships of two different nets (DESIGN.md f14) -- brl_model_rows by player id against its NumPy restatement,
brl_duplicate_match with nets by player id against the [n, 2] call and the host loop, brl_evaluate_match's partner mode
against the unflagged call and the host loops, the roll-out's partner sub-step, cross-play, and ppo.train /
train_population with a fixed partner."""
import numpy as np
import pytest
import torch

from tests import helpers as H
from tests.test_partner_host import ref_player_grouping

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FORCE_FUSED, FORCE_LAYERS = 1 << 30, 1 << 29  # BRL_F_TUNE_MLP_FUSED, BRL_F_TUNE_MLP_LAYERS (include/brl_b200.h)


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


def _pin_host_path(monkeypatch, tune):
    """make the host loop's listed forwards take the path `tune` pins"""
    from brl_b200 import ops
    orig = ops.policy_act_rows
    monkeypatch.setattr(ops, "policy_act_rows", lambda *a, **kw: orig(*a, **{**kw, "tune": kw.get("tune", 0) | tune}))


# ---- brl_model_rows with BRL_F_PLAYER_MODELS --------------------------------------------------------------------------
def _grouping_outputs(n, M):
    from brl_b200 import ops
    cap = ops.model_rows_capacity(n, M)
    poison = lambda *shape: torch.full(shape, -1, dtype=torch.int32, device=DEV)  # noqa: E731 -- 0xFF bytes
    return poison(max(cap, 1)), poison(M), poison(M + 1), poison(max(cap // 256, 1))


def _model_rows(player, done, env_models, M):
    from brl_b200 import ops
    rows, counts, offsets, block_model = _grouping_outputs(player.shape[0], M)
    ops.model_rows(player, done, env_models, rows, counts, offsets, block_model)
    torch.cuda.synchronize()
    return rows.cpu().numpy(), counts.cpu().numpy(), offsets.cpu().numpy(), block_model.cpu().numpy()


def _assert_grouping(got, want, M):
    """counts, offsets and block ids exactly; each group's rows as a set (their order inside a group is the order in which
    the warps' atomics arrive), then -1 padding"""
    rows, counts, offsets, block_model = got
    w_counts, w_offsets, w_rows, w_blocks = want
    assert (counts == w_counts).all() and (offsets == w_offsets).all()
    if offsets[M] < 0:
        return
    for m in range(M):
        lo = offsets[m]
        assert sorted(rows[lo:lo + counts[m]].tolist()) == w_rows[m]
        assert (rows[lo + counts[m]:offsets[m + 1]] == -1).all()
    assert (block_model[:offsets[M] // 256] == w_blocks).all()


@pytest.mark.parametrize("n", [0, 1, 255, 4097, 65536 + 333])
def test_player_grouping_equals_the_numpy_restatement_and_the_team_call(n):
    g = np.random.default_rng(n)
    M = 5
    player = g.integers(0, 4, n).astype(np.int8)
    done = (g.random(n) < 0.2).astype(np.uint8)
    ids = g.integers(0, M, (n, 4)).astype(np.int32)
    t = lambda a: torch.as_tensor(a, device=DEV).contiguous()  # noqa: E731
    if n == 0:
        got = _model_rows(t(player), t(done), t(ids), M)
        assert (got[1] == 0).all() and (got[2] == 0).all()
        return
    _assert_grouping(_model_rows(t(player), t(done), t(ids), M), ref_player_grouping(player, done, ids, M), M)
    # partners on the same net: the by-player call groups exactly as the by-team call
    team = ids[:, [0, 2]]
    same = team[:, [0, 0, 1, 1]]
    got4, got2 = _model_rows(t(player), t(done), t(same), M), _model_rows(t(player), t(done), t(team), M)
    for a, b in zip(got4[1:], got2[1:]):
        assert (a == b).all()
    _assert_grouping(got4, ref_player_grouping(player, done, same, M), M)
    _assert_grouping(got2, ref_player_grouping(player, done, same, M), M)
    # a live env whose acting player's id is outside [0, M): offsets[M] = -1
    bad = ids.copy()
    i = int(np.flatnonzero(done == 0)[0])
    bad[i, player[i]] = M
    assert _model_rows(t(player), t(done), t(bad), M)[2][M] == -1


# ---- brl_duplicate_match with BRL_F_PLAYER_MODELS -----------------------------------------------------------------------
def _play(env, n, nets, models, tune=0, single_bf16=False):
    """one brl_duplicate_match over `nets` with env_models `models` ([n, 2] or [n, 4], the same row for every env)"""
    from brl_b200 import ops, random as brandom
    from brl_b200.evaluation import _MatchBuffers
    from brl_b200.models import make_forward_pass
    width = len(models)
    b = _MatchBuffers(n, len(nets), 0, DEV, with_models=True, with_tables=True, players=width == 4)
    fp = make_forward_pass("relu", "DeepMind")
    size = ops._lib.load().brl_mlp_packed_bytes()
    for m, p in enumerate(nets):
        fp.pack_into(p, b.pool[m, :size])
    _, sub = brandom.split(brandom.PRNGKey(n))
    b.keys.copy_(env.make_keys(sub, n))
    b.env_models.copy_(torch.tensor(models, dtype=torch.int32, device=DEV).expand(n, width))
    b.cum_return.fill_(float("nan"))
    b.play(env, single_bf16, tune)
    torch.cuda.synchronize()
    assert int(b.status[0]) == 0
    return b


@pytest.mark.parametrize("single_bf16", [False, True])
@pytest.mark.parametrize("n", [1, 100, 4096, 10000])
def test_partners_on_one_net_equal_the_team_match(n, single_bf16):
    env = _env()
    nets = [H.seeded_params(700 + k, DEV) for k in range(3)]
    by_player = _play(env, n, nets, [0, 0, 2, 2], single_bf16=single_bf16)
    by_team = _play(env, n, nets, [0, 2], single_bf16=single_bf16)
    assert torch.equal(by_player.cum_return, by_team.cum_return) and torch.equal(by_player.sums, by_team.sums)
    for ta, tb in zip(by_player.tables, by_team.tables):
        for f in ("terminated", "rewards", "last_bid", "last_bidder", "call_x", "call_xx"):
            assert torch.equal(getattr(ta, f), getattr(tb, f)), f


@pytest.mark.parametrize("precision, tune", [("tc", 0), ("tc-bf16", 0), ("tc", FORCE_LAYERS), ("tc", FORCE_FUSED)],
                         indirect=["precision"])
@pytest.mark.parametrize("n", [1, 100, 4096, 10000])
def test_four_nets_equal_the_host_loop_with_per_player_nets(n, precision, tune, monkeypatch):
    from brl_b200 import random as brandom
    from brl_b200.evaluation import _make_device_pair_matches, make_simple_duplicate_evaluate
    from brl_b200.models import make_forward_pass
    if tune:
        _pin_host_path(monkeypatch, tune)
    env = _env()
    a, b, c, d = (H.seeded_params(710 + k, DEV) for k in range(4))
    key = brandom.PRNGKey(31 + n)
    host_cum = {}
    want = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)(
        a, c, key, team1_partner=b, team2_partner=d)
    matches = _make_device_pair_matches(env, make_forward_pass("relu", "DeepMind", precision=precision), n, 1 << 20, tune)
    got = matches([(0, 1, 2, 3)], key, params_list=[a, b, c, d], cum_returns=host_cum)
    np.testing.assert_allclose(got[0], want[0], rtol=1e-12, atol=0)
    assert torch.equal(host_cum[(0, 1, 2, 3)], want[3])


# ---- brl_evaluate_match with BRL_F_EVAL_PARTNER ----------------------------------------------------------------------------
def _assert_log_info(got, want):
    assert len(got) == len(want)
    for g, w in zip(got, want):
        np.testing.assert_allclose(np.asarray(g, dtype=np.float64), np.asarray(w, dtype=np.float64), rtol=1e-12, atol=0)


def _host_acc(monkeypatch):
    from brl_b200 import ops
    seen = {}
    orig = ops.eval_summary

    def spy(acc, cum_return, *a, **kw):
        seen["acc"], seen["cum_return"] = acc.clone(), cum_return.clone()
        return orig(acc, cum_return, *a, **kw)
    monkeypatch.setattr(ops, "eval_summary", spy)
    return seen


@pytest.mark.parametrize("precision", ["tc", "tc-bf16"], indirect=True)
@pytest.mark.parametrize("duplicate", [True, False])
@pytest.mark.parametrize("game_mode", ["competitive", "free-run"])
@pytest.mark.parametrize("n", [100, 4097])
def test_full_evaluation_with_a_partner(n, game_mode, duplicate, precision, monkeypatch):
    from brl_b200 import random as brandom
    from brl_b200.evaluation import make_device_evaluate, make_evaluate
    env = _env()
    actor, opp, partner = (H.seeded_params(720 + k, DEV) for k in range(3))
    key = brandom.PRNGKey(40 + n)
    dev_eval = make_device_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, game_mode, duplicate=duplicate,
                                    team2_params=opp)
    plain = dev_eval(actor, key)
    plain_acc, plain_cum = dev_eval.buffers.acc.clone(), dev_eval.buffers.cum_return.clone()
    same = dev_eval(actor, key, partner_params=actor)          # partner = actor: the unflagged call's results
    assert dev_eval.buffers.partner
    assert torch.equal(dev_eval.buffers.acc, plain_acc) and torch.equal(dev_eval.buffers.cum_return, plain_cum)
    _assert_log_info(same[0] if duplicate else same[1], plain[0] if duplicate else plain[1])
    seen = _host_acc(monkeypatch)
    want = make_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, game_mode, duplicate=duplicate,
                         team2_params=opp)(actor, key, partner_params=partner)
    got = dev_eval(actor, key, partner_params=partner)
    assert torch.equal(dev_eval.buffers.acc, seen["acc"]) and torch.equal(dev_eval.buffers.cum_return, seen["cum_return"])
    assert not torch.equal(dev_eval.buffers.acc, plain_acc)
    if duplicate:
        for t_got, t_want in zip(got[1:], want[1:]):
            for f in t_want._fields:
                assert torch.equal(getattr(t_got, f), getattr(t_want, f)), f
        _assert_log_info(got[0], want[0])
    else:
        for k in ("_packed", "observation", "_mask_u8", "rewards", "_terminated_u8", "current_player"):
            assert torch.equal(getattr(got[0], k), getattr(want[0], k)), k
        _assert_log_info(got[1], want[1])


@pytest.mark.parametrize("precision", ["tc", "tc-bf16"], indirect=True)
@pytest.mark.parametrize("n", [1, 300, 4097])
def test_simple_evaluation_with_a_partner(n, precision):
    from brl_b200 import random as brandom
    from brl_b200.evaluation import make_device_simple_evaluate, make_simple_evaluate
    env = _env()
    actor, opp, partner = (H.seeded_params(730 + k, DEV) for k in range(3))
    key = brandom.PRNGKey(50 + n)
    dev_eval = make_device_simple_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, team2_params=opp)
    plain = float(dev_eval(actor, key))
    plain_R = dev_eval.buffers.cum_return.clone()
    assert float(dev_eval(actor, key, partner_params=actor)) == plain
    assert torch.equal(dev_eval.buffers.cum_return, plain_R)
    trace = []
    want = make_simple_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, team2_params=opp)(
        actor, key, trace=trace, partner_params=partner)
    got = dev_eval(actor, key, partner_params=partner)
    assert trace[-1][0] == "R" and torch.equal(dev_eval.buffers.cum_return, trace[-1][1])
    assert float(got) == float(want)


# ---- the roll-out's partner sub-step -----------------------------------------------------------------------------------
def _runner(env, params, keys):
    from brl_b200 import random as brandom
    state = env.init(keys)
    return (params, None, state, state.observation, torch.zeros((), dtype=torch.int64, device=DEV), brandom.PRNGKey(9))


def _roll(roll_out, runner, opp, **kw):
    runner, traj = roll_out(runner, opp, **kw)
    torch.cuda.synchronize()
    st = runner[2]
    final = (st._packed.clone(), st.observation.clone(), st._mask_u8.clone(), st.current_player.clone())
    return {k: getattr(traj, k).clone() for k in traj._fields}, final, int(runner[4])


def _same_roll(a, b):
    return all(torch.equal(a[0][k], b[0][k]) for k in a[0]) and all(torch.equal(x, y) for x, y in zip(a[1], b[1])) and a[2] == b[2]


@pytest.mark.parametrize("game_mode", ["competitive", "free-run"])
def test_roll_out_with_a_partner(game_mode):
    from brl_b200.models import make_forward_pass
    from brl_b200.roll_out import make_roll_out
    env = _env(seed=8)
    n, T = 4096, 6
    cfg = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode=game_mode, num_steps=T,
               reward_scale=7600.0)
    actor, opp, partner = (H.seeded_params(740 + k, DEV) for k in range(3))
    fp, partner_fp = make_forward_pass("relu", "DeepMind"), make_forward_pass("relu", "DeepMind")
    ro = make_roll_out(dict(cfg), env, fp, fp, partner_forward_pass=partner_fp)
    keys = env.make_keys(5, n)
    plain = _roll(ro, _runner(env, actor, keys), opp, graph_seeding=True)
    # partner = actor: the unpartnered trajectory and final state, on the plain path and on the graph path
    assert _same_roll(_roll(ro, _runner(env, actor, keys), opp, partner_params=actor, graph_seeding=True), plain)
    g_plain = _roll(ro, _runner(env, actor, keys), opp)
    assert _same_roll(g_plain, plain)
    assert _same_roll(_roll(ro, _runner(env, actor, keys), opp, partner_params=actor), g_plain)
    # a distinct partner: sub-step 3 is the partner's (traced), and the graph path replays the seeded plain path
    trace = []
    _roll(ro, _runner(env, actor, keys), opp, partner_params=partner, trace=trace)
    assert len(trace) == 4 * T
    seeded = _roll(ro, _runner(env, actor, keys), opp, partner_params=partner, graph_seeding=True)
    assert not _same_roll(seeded, plain)
    for _ in range(2):
        assert _same_roll(_roll(ro, _runner(env, actor, keys), opp, partner_params=partner), seeded)
    assert _same_roll(_roll(ro, _runner(env, actor, keys), opp), g_plain)  # the unpartnered graph is untouched


# ---- cross-play ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1, 3, 8])
def test_crossplay(M):
    from brl_b200 import random as brandom
    from brl_b200.evaluation import (make_crossplay_evaluate, make_device_duplicate_evaluate,
                                     make_simple_duplicate_evaluate)
    env = _env()
    n = 100
    nets = [H.seeded_params(750 + k, DEV) for k in range(M)]
    c, d = H.seeded_params(790, DEV), H.seeded_params(791, DEV)
    key = brandom.PRNGKey(7)
    cums = {}
    stats, imp = make_crossplay_evaluate(env, "relu", "DeepMind", n)(nets, (c, d), key, cum_returns=cums)
    assert imp.shape == (M, M) and sorted(stats) == [(a, b) for a in range(M) for b in range(M)]
    chunked = make_crossplay_evaluate(env, "relu", "DeepMind", n, max_envs=2 * n + 37)(nets, (c, d), key)
    assert chunked[0] == stats and (chunked[1] == imp).all()
    host = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)
    for (a, b) in ([(a, b) for a in range(M) for b in range(M)] if M <= 3 else [(0, 0), (M - 1, 2), (3, 5)]):
        want = host(nets[a], c, key, team1_partner=nets[b], team2_partner=d)
        np.testing.assert_allclose(stats[(a, b)], want[0], rtol=1e-12, atol=0)
        assert torch.equal(cums[(a, b)], want[3]) and imp[a, b] == stats[(a, b)][0]
    diag = make_crossplay_evaluate(env, "relu", "DeepMind", n)(nets, (c, c), key)[0]
    dup = make_device_duplicate_evaluate(env, "relu", "DeepMind", n)
    for a in range(M):
        assert diag[(a, a)] == tuple(dup(nets[a], c, key)[0])


def test_device_duplicate_evaluate_with_a_partner():
    from brl_b200 import random as brandom
    from brl_b200.evaluation import make_device_duplicate_evaluate, make_simple_duplicate_evaluate
    env = _env()
    n = 4097
    a, b, c = (H.seeded_params(760 + k, DEV) for k in range(3))
    key = brandom.PRNGKey(3)
    dup = make_device_duplicate_evaluate(env, "relu", "DeepMind", n)
    plain, same = dup(a, c, key), dup(a, c, key, team1_partner=a)
    assert plain[0] == same[0] and torch.equal(plain[3], same[3])
    want = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)(a, c, key, team1_partner=b)
    got = dup(a, c, key, team1_partner=b)
    np.testing.assert_allclose(got[0], want[0], rtol=1e-12, atol=0)
    assert torch.equal(got[3], want[3])
    for t_got, t_want in zip(got[1:3], want[1:3]):
        for f in t_want._fields:
            assert torch.equal(getattr(t_got, f), getattr(t_want, f)), f


# ---- ppo.train / train_population with a fixed partner -------------------------------------------------------------------
def _train_config(tmp_path, name, **kw):
    base = dict(num_envs=128, num_steps=4, minibatch_size=128, update_epochs=2, total_timesteps=128 * 4 * 3, hash_size=20,
                num_eval_envs=64, num_prioritized_envs=32, num_eval_step=2, save_model=False, log_path=str(tmp_path), exp_name=name)
    base.update(kw)
    return base


def _save_net(tmp_path, seed, name):
    from brl_b200 import ppo
    path = str(tmp_path / f"{name}.pkl")
    ppo.save_params(H.seeded_params(seed, DEV), path)
    return path


def _tables():
    from brl_b200.deals import synthetic_deal_table
    return [synthetic_deal_table(300, seed=k) for k in range(2)], synthetic_deal_table(200, seed=9)


def _same_runs(a, b):
    from brl_b200.models import params_to_numpy
    (runner_a, logs_a), (runner_b, logs_b) = a, b
    assert len(logs_a) == len(logs_b)
    for la, lb in zip(logs_a, logs_b):
        keys = sorted(x for x in lb if not x.startswith("time/"))
        assert keys == sorted(x for x in la if not x.startswith("time/"))
        for x in keys:
            np.testing.assert_allclose(la[x], lb[x], rtol=1e-12, atol=0, err_msg=x)
    pa, pb = params_to_numpy(runner_a[0]), params_to_numpy(runner_b[0])
    assert all((pa[x] == pb[x]).all() for x in pa)


def test_train_with_partner_model_path_none_equals_train_without(tmp_path):
    from brl_b200 import ppo, random as brandom
    tables, eval_table = _tables()
    plain = ppo.train(_train_config(tmp_path, "a", lr=1e-4), brandom.PRNGKey(3), tables=tables, eval_table=eval_table, device=DEV)
    spelled = ppo.train(_train_config(tmp_path, "b", lr=1e-4, partner_model_path=None), brandom.PRNGKey(3), tables=tables,
                        eval_table=eval_table, device=DEV)
    _same_runs(spelled, plain)


def test_partnered_training_evaluates_with_the_partner(tmp_path, monkeypatch):
    """the partnered run's train/score, imp_opp_* and eval/* (log_par's too) equal the host evaluators' given the partner"""
    from brl_b200 import ppo, random as brandom
    tables, eval_table = _tables()
    partner = _save_net(tmp_path, 770, "partner")
    cfg = _train_config(tmp_path, "p", lr=1e-4, partner_model_path=partner, num_eval_envs=300, num_prioritized_envs=100,
                        num_eval_step=1)

    def run(**kw):
        return ppo.train(dict(cfg, **kw), brandom.PRNGKey(5), tables=tables, eval_table=eval_table, device=DEV,
                         eval_opp_params=H.seeded_params(771, DEV))
    with monkeypatch.context() as m:
        m.setattr(ppo, "make_evaluators", H.host_evaluators)
        host = run()
    dev = run()
    plain = run(partner_model_path=None)
    keys = [k for k in host[1][0] if k.startswith(("train/score", "train/imp_opp", "eval/"))]
    assert "eval/IMP_reward" in keys and "train/imp_opp_after" in keys
    for h, d in zip(host[1], dev[1]):
        for k in keys:
            np.testing.assert_allclose(d[k], h[k], rtol=1e-12, atol=0, err_msg=k)
    assert any(plain[1][0][k] != dev[1][0][k] for k in keys)
    par = run(log_par=True)  # log_par's match is the partnered eval/* match
    assert all(np.isfinite(log["eval/imp_vs_par"]) for log in par[1])
    _same_runs((par[0], [{k: v for k, v in log.items() if "par" not in k} for log in par[1]]), dev)


def test_train_population_with_partners_equals_solo_runs(tmp_path):
    from brl_b200 import ppo, random as brandom
    tables, eval_table = _tables()
    partner = _save_net(tmp_path, 772, "partner")

    def configs(tag):
        return [_train_config(tmp_path, f"{tag}0", seed=0, lr=1e-4, partner_model_path=partner),
                _train_config(tmp_path, f"{tag}1", seed=1, lr=3e-4, ent_coef=0.01)]
    pop = ppo.train_population(configs("p"), [brandom.PRNGKey(20), brandom.PRNGKey(21)], tables=tables,
                               eval_table=eval_table, device=DEV)
    for k, cfg in enumerate(configs("s")):
        _same_runs(pop[k], ppo.train(cfg, brandom.PRNGKey(20 + k), tables=tables, eval_table=eval_table, device=DEV))


def test_partnered_roll_out_replays_through_the_oracle():
    """free-run (the partner's sub-step is an argmax): every traced sub-step replays through the oracle env into the recorded
    done, reward and next observation, and sub-step 3's action is the partner's masked argmax on the oracle's observation
    (the actor's would differ)"""
    from brl_b200 import random as brandom
    from brl_b200.deals import synthetic_deal_table
    from brl_b200.env import BridgeBidding
    from brl_b200.models import make_forward_pass, params_to_numpy
    from brl_b200.roll_out import make_roll_out
    from oracle import oracle as orc
    table = synthetic_deal_table(3000, seed=2)
    env = BridgeBidding(table=table, device=DEV)
    n, T = 512, 8
    config = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode="free-run", num_steps=T,
                  reward_scale=7600.0)
    fp = make_forward_pass("relu", "DeepMind")
    actor, opp, partner = (H.seeded_params(780 + k, DEV) for k in range(3))
    keys = env.make_keys(77, n)
    state = env.init(keys)
    runner = (actor, None, state, state.observation, torch.zeros((), dtype=torch.int64, device=DEV), brandom.PRNGKey(3))
    trace = []
    runner2, traj = make_roll_out(config, env, fp, fp, partner_forward_pass=make_forward_pass("relu", "DeepMind"))(
        runner, opp, partner_params=partner, trace=trace)
    assert len(trace) == 4 * T
    ref = orc.OracleEnv(table, n)
    ref.init(keys.cpu().numpy().view(np.uint64))
    e = ref.export()
    nets = {"partner": params_to_numpy(partner), "actor": params_to_numpy(actor)}
    agree = {"partner": 0, "actor": 0}
    decided = 0
    for t in range(T):
        who = e["current_player"].copy()
        rew, term = np.zeros((n, 4), np.float32), np.zeros(n, np.uint8)
        for k in range(4):
            a = trace[4 * t + k].cpu().numpy()
            if k == 2:  # the partner's slot: its masked argmax on this observation
                mask = e["legal_action_mask"].astype(bool)
                live = ~e["terminated"].astype(bool)
                for name, p in nets.items():
                    logits, _ = orc.mlp_forward(p, e["observation"].astype(np.float32))
                    ml = np.where(mask, logits, -np.inf)
                    top2 = np.sort(ml, axis=1)[:, -2:]
                    clear = live & (top2[:, 1] - top2[:, 0] > 1e-3)
                    agree[name] += int((ml.argmax(1) == a)[clear].sum())
                    if name == "partner":
                        decided += int(clear.sum())
            ref.step(a, autoreset=True)
            e = ref.export()
            rew += e["rewards"]
            term |= e["terminated"]
        assert (traj.done[t].cpu().numpy() == term.astype(bool)).all(), t
        assert (traj.reward[t].cpu().numpy() == rew[np.arange(n), who] / np.float32(7600.0)).all(), t
        obs_next = traj.obs[t + 1] if t + 1 < T else runner2[3]
        assert (obs_next.float().cpu().numpy() == e["observation"]).all(), t
    assert decided > 1000 and agree["partner"] == decided and agree["actor"] < decided
