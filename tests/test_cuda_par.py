"""GPU: brl_par against the par reference (tests/par_ref.py) bit for bit, brl_gather_reward_par, and the "par_imp" roll-out
against the "score" roll-out from the same runner state and keys."""
import functools

import numpy as np
import pytest
import torch

from tests import helpers as H
from tests import par_ref as P

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@functools.lru_cache(maxsize=None)
def _dd_of(table_id):
    from brl_b200.deals import unpack_deal_table
    return unpack_deal_table(_TABLES[table_id])[1]


_TABLES = {}


def _table(name):
    if name not in _TABLES:
        if name == "real":
            _TABLES[name] = H.load_boards()["table"]
        else:
            from brl_b200.deals import synthetic_deal_table
            _TABLES[name] = synthetic_deal_table(100_000, seed={"synth_a": 3, "synth_b": 4}[name])
    return _TABLES[name]


@functools.lru_cache(maxsize=None)
def _oracle(table_id, deal, dealer, vns, vew):
    return P.par(_dd_of(table_id)[deal], dealer, vns, vew)


def _device_par(env, state):
    """ops.par into outputs poisoned with 0xFF"""
    from brl_b200 import ops
    n = state.num_envs
    par = torch.full((n, 4), -1, dtype=torch.int32, device=DEV).view(torch.float32)
    contract = torch.full((n,), -1, dtype=torch.int32, device=DEV)
    ops.par(state._packed, env.table, par, contract)
    torch.cuda.synchronize()
    return par.cpu().numpy(), contract.cpu().numpy()


def _check(table_id, env, state, rows=None):
    deal, dealer, seat, vul = (state._f(k).cpu().numpy() for k in ("deal", "dealer", "shuffled_players", "vul"))
    par, contract = _device_par(env, state)
    rows = np.arange(state.num_envs) if rows is None else rows
    for i in rows:
        v, c = _oracle(table_id, int(deal[i]), int(dealer[i]), int(vul[i, 0]), int(vul[i, 1]))
        assert contract[i] == c, (i, contract[i], c)
        assert (par[i] == P.par_by_player(v, seat[i])).all(), (i, par[i], v)
    return deal, dealer, vul, par, contract


def test_par_of_the_real_boards_under_every_dealer_and_vulnerability():
    from brl_b200.env import BridgeBidding
    table = _table("real")
    env = BridgeBidding(table=table, device=DEV)
    n = len(table)
    rng = np.random.default_rng(0)
    deal = np.tile(np.arange(n), 16)
    combo = np.repeat(np.arange(16), n)
    dealer, vns, vew = combo % 4, (combo >> 2) & 1, (combo >> 3) & 1
    seating = H.SEATINGS[rng.integers(0, 8, len(deal))]
    state = env.init_from(deal, dealer, vns, vew, seating)
    _check("real", env, state)


@pytest.mark.parametrize("n", [1, 255, 8192, 1 << 20])
@pytest.mark.parametrize("table_id", ["synth_a", "synth_b"])
def test_par_of_synthetic_boards_from_init_and_duplicate_init(table_id, n):
    """every env against the reference up to 8,192 envs; at 1,048,576 envs a sample of 4,096 against the reference, and every
    env against the envs that share its board, dealer and vulnerability"""
    from brl_b200.duplicate import duplicate_init
    from brl_b200.env import BridgeBidding
    env = BridgeBidding(table=_table(table_id), device=DEV)
    state = env.init(env.make_keys(n * 7 + 1, n))
    rows = None if n <= 8192 else np.random.default_rng(n).choice(n, 4096, replace=False)
    a = _check(table_id, env, state, rows)
    b = _check(table_id, env, duplicate_init(state), rows)
    for x, y in zip(a[:3], b[:3]):  # the same boards at the other table
        assert (x == y).all()
    assert (a[4] == b[4]).all() and (a[3] == -b[3]).all()  # teams swap seats: the par by player id flips sign
    if n > 8192:
        deal, dealer, vul, par, contract = a
        key = ((deal.astype(np.int64) * 4 + dealer) * 2 + vul[:, 0]) * 2 + vul[:, 1]
        ns = np.where(state._f("shuffled_players").cpu().numpy()[:, 0] >> 1 == 0, par[:, 0], -par[:, 0])
        order = np.argsort(key, kind="stable")
        same = key[order][1:] == key[order][:-1]
        assert same.sum() > 1000
        assert (ns[order][1:][same] == ns[order][:-1][same]).all()
        assert (contract[order][1:][same] == contract[order][:-1][same]).all()


def test_gather_reward_par_and_its_count():
    from brl_b200 import ops
    rng = np.random.default_rng(5)
    n = 10_000
    rewards = (rng.integers(-760, 761, n) * 10).astype(np.float32)
    par = (rng.integers(-222, 223, n) * 10).astype(np.float32)
    sign = rng.choice([1.0, -1.0], n).astype(np.float32)
    r4 = np.stack([rewards, rewards, -rewards, -rewards], 1) * sign[:, None]
    p4 = np.stack([par, par, -par, -par], 1) * sign[:, None]
    actor = rng.integers(0, 4, n).astype(np.int8)
    done = (rng.random(n) < 0.3).astype(np.uint8)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=DEV)  # noqa: E731
    out = torch.full((n,), float("nan"), device=DEV)
    count = torch.full((1,), 5, dtype=torch.int64, device=DEV)
    ops.gather_reward_par(t(r4), t(actor), t(p4), t(done), out, count=count)
    want = np.array([P.par_reward(r4[i, actor[i]], p4[i, actor[i]]) if done[i] else 0.0 for i in range(n)], np.float32)
    assert (out.cpu().numpy() == want).all()
    assert int(count) == 5 + int(done.sum())
    out2 = torch.empty_like(out)
    ops.gather_reward_par(t(r4), t(actor), t(p4), t(done), out2)  # without the count
    assert torch.equal(out, out2)


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


@pytest.mark.parametrize("graph", [False, True])
def test_par_imp_roll_out_equals_the_score_roll_out_but_for_the_reward(graph, monkeypatch):
    from brl_b200 import ops
    from brl_b200.deals import synthetic_deal_table, unpack_deal_table
    from brl_b200.env import BridgeBidding
    from brl_b200.models import init_params, make_forward_pass
    from brl_b200.roll_out import make_roll_out
    table = synthetic_deal_table(5000, seed=8)
    env = BridgeBidding(table=table, device=DEV)
    n, T = 4096, 8
    base = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode="competitive",
                num_steps=T, reward_scale=7600.0)
    params, opp = H.seeded_params(101, DEV), init_params(102, DEV)
    fp = make_forward_pass("relu", "DeepMind")
    score_ro = make_roll_out(dict(base), env, fp, fp)
    par_ro = make_roll_out(dict(base, reward_mode="par_imp"), env, fp, fp)
    keys = env.make_keys(5, n)

    # the reference run: par mode on the plain path with the graph's seeds, recording every step's pre-step par, the board
    # fields of the pre-step state and the actor
    recorded, actors = [], []
    real_par, real_gather = ops.par, ops.gather_reward_par

    def recording_par(state_packed, tab, out, contract=None):
        real_par(state_packed, tab, out, contract)
        f = ops.state_fields(state_packed)
        recorded.append((out.clone(), {k: f[k].clone() for k in ("deal", "dealer", "vul", "shuffled_players")}))

    def recording_gather(rewards, actor, par, done, out, count=None):
        actors.append(actor.clone())
        real_gather(rewards, actor, par, done, out, count=count)

    monkeypatch.setattr(ops, "par", recording_par)
    monkeypatch.setattr(ops, "gather_reward_par", recording_gather)
    ref_par, ref_final, ref_count = _roll(par_ro, _runner(env, params, keys), opp, graph_seeding=True)
    monkeypatch.setattr(ops, "par", real_par)
    monkeypatch.setattr(ops, "gather_reward_par", real_gather)
    assert len(recorded) == len(actors) == T
    ref_score, score_final, score_count = _roll(score_ro, _runner(env, params, keys), opp, graph_seeding=True)
    for k in ("obs", "legal_action_mask", "action", "done", "log_prob", "value"):
        assert torch.equal(ref_par[k], ref_score[k]), k
    assert all(torch.equal(a, b) for a, b in zip(ref_final, score_final)) and ref_count == score_count

    # reward = IMP(score - par) / 24 on every done (t, env), 0 elsewhere; par from the deal the pre-step state holds
    dd = unpack_deal_table(table)[1]
    done = ref_par["done"].cpu().numpy()
    assert done.sum() > 1000
    score = np.rint(ref_score["reward"].cpu().numpy().astype(np.float64) * 7600.0)  # the actor's score, exact
    got = ref_par["reward"].cpu().numpy()
    for t in range(T):
        par_t, f = recorded[t]
        par_t, actor = par_t.cpu().numpy(), actors[t].cpu().numpy().astype(np.int64)
        deal, dealer, vul, seat = (f[k].cpu().numpy() for k in ("deal", "dealer", "vul", "shuffled_players"))
        want = np.zeros(n, np.float32)
        for i in np.flatnonzero(done[t]):
            v, _ = P.par(dd[deal[i]], int(dealer[i]), int(vul[i, 0]), int(vul[i, 1]))
            lay = P.par_by_player(v, seat[i])
            assert (par_t[i] == lay).all()
            want[i] = P.par_reward(score[t, i], lay[actor[i]])
        assert (got[t] == want).all(), t

    if graph:  # the CUDA-graph path replays the reference runs bit for bit, in both modes, and keeps its score graph
        for _ in range(2):
            g_par, g_final, _ = _roll(par_ro, _runner(env, params, keys), opp)
            g_score, gs_final, _ = _roll(score_ro, _runner(env, params, keys), opp)
        for k in ref_par:
            assert torch.equal(g_par[k], ref_par[k]), k
            assert torch.equal(g_score[k], ref_score[k]), k
        assert all(torch.equal(a, b) for a, b in zip(g_final, ref_final))


def _swap_seats(seat):
    """table B's seating (duplicate_init): the players of seats N/E and of seats S/W trade places"""
    return seat[:, [1, 0, 3, 2]]


def _par_statistics_ref(eval_env, init_state, a, b):
    """par_statistics restated on the host from the reference par"""
    from brl_b200.deals import unpack_deal_table
    dd = unpack_deal_table(eval_env.table_np)[1]
    deal, dealer, vul, seat = (init_state._f(k).cpu().numpy() for k in ("deal", "dealer", "vul", "shuffled_players"))
    imps, hits = [], []
    for info, seats in ((a, seat), (b, _swap_seats(seat))):
        rew, bid, bidder = info.rewards.cpu().numpy(), info.last_bid.cpu().numpy(), info.last_bidder.cpu().numpy()
        for i in range(len(deal)):
            v, c = P.par(dd[deal[i]], int(dealer[i]), int(vul[i, 0]), int(vul[i, 1]))
            imps.append(P.imp(int(rew[i, 0]) - int(P.par_by_player(v, seats[i])[0])))
            if bid[i] < 0 or c < 0:
                hits.append(bid[i] < 0 and c < 0)
            else:
                side = int(np.flatnonzero(seats[i] == bidder[i])[0]) & 1
                hits.append(bid[i] == (c & 0xFF) and side == (c >> 8) & 1)
    x = np.array(imps, np.float64)
    se = x.std(ddof=1) / np.sqrt(len(x)) if len(x) > 1 else float("nan")
    return x.mean(), se, np.abs(x).mean(), np.mean(hits)


@pytest.mark.parametrize("game_mode", ["competitive", "free-run"])
@pytest.mark.parametrize("n", [1, 100, 10_000])
def test_par_statistics_of_a_device_duplicate_match(n, game_mode):
    from brl_b200 import random as brandom
    from brl_b200.deals import synthetic_deal_table
    from brl_b200.env import BridgeBidding
    from brl_b200.evaluation import make_device_evaluate, par_statistics
    eval_env = BridgeBidding(table=synthetic_deal_table(3000, seed=21), device=DEV)
    evaluate = make_device_evaluate(eval_env, "relu", "DeepMind", "relu", "DeepMind", None, n, game_mode, duplicate=True,
                                    team2_params=H.seeded_params(32, DEV))
    _, a, b = evaluate(H.seeded_params(31, DEV), brandom.PRNGKey(n))
    init_state = eval_env.init(evaluate.buffers.keys)
    got = par_statistics(eval_env, init_state, a, b)
    mean, se, abs_mean, rate = _par_statistics_ref(eval_env, init_state, a, b)
    assert got["imp_vs_par"][0] == pytest.approx(mean, rel=1e-12, abs=1e-12)
    if n > 1:
        assert got["imp_vs_par"][1] == pytest.approx(se, rel=1e-9, abs=1e-12)
    assert got["abs_imp_vs_par"] == pytest.approx(abs_mean, rel=1e-12, abs=1e-12)
    assert got["par_contract_rate"] == pytest.approx(rate, rel=1e-12, abs=1e-12)
    if n == 10_000:
        assert 0.0 < got["abs_imp_vs_par"]


def _train_config(tmp_path, name, **kw):
    base = dict(num_envs=128, num_steps=4, minibatch_size=128, update_epochs=2, total_timesteps=128 * 4 * 3, hash_size=20,
                num_eval_envs=64, num_prioritized_envs=32, num_eval_step=2, save_model=False, log_path=str(tmp_path), exp_name=name)
    base.update(kw)
    return base


def _tables():
    from brl_b200.deals import synthetic_deal_table
    return [synthetic_deal_table(300, seed=k) for k in range(2)], synthetic_deal_table(200, seed=9)


PAR_KEYS = {"eval/imp_vs_par", "eval/abs_imp_vs_par", "eval/par_contract_rate"}


def test_train_with_the_default_reward_and_log_settings_spelled_out_equals_train_without(tmp_path):
    from brl_b200 import ppo, random as brandom
    from brl_b200.models import params_to_numpy
    tables, eval_table = _tables()
    runs = [ppo.train(_train_config(tmp_path, name, lr=1e-4, **kw), brandom.PRNGKey(3), tables=tables, eval_table=eval_table,
                      device=DEV) for name, kw in (("a", {}), ("b", dict(reward_mode="score", log_par=False)))]
    (ra, la), (rb, lb) = runs
    assert len(la) == len(lb) == 3
    for x, y in zip(la, lb):
        assert {k: v for k, v in x.items() if not k.startswith("time/")} == {k: v for k, v in y.items() if not k.startswith("time/")}
        assert not PAR_KEYS & set(x)
    pa, pb = params_to_numpy(ra[0]), params_to_numpy(rb[0])
    assert all((pa[k] == pb[k]).all() for k in pa)


def test_log_par_adds_the_par_statistics_of_the_eval_match(tmp_path, monkeypatch):
    from brl_b200 import ppo, random as brandom
    from brl_b200.models import params_to_numpy
    tables, eval_table = _tables()
    seen = []
    real = ppo.par_statistics

    def recording(eval_env, init_state, a, b):
        got = real(eval_env, init_state, a, b)
        seen.append((got, _par_statistics_ref(eval_env, init_state, a, b)))
        return got

    monkeypatch.setattr(ppo, "par_statistics", recording)
    runner_p, logs_p = ppo.train(_train_config(tmp_path, "p", lr=1e-4, log_par=True), brandom.PRNGKey(3), tables=tables,
                                 eval_table=eval_table, device=DEV)
    runner_q, logs_q = ppo.train(_train_config(tmp_path, "q", lr=1e-4), brandom.PRNGKey(3), tables=tables,
                                 eval_table=eval_table, device=DEV)
    assert len(seen) == 2  # iterations 0 and 2 play the eval/* match
    it = iter(seen)
    for i, (lp, lq) in enumerate(zip(logs_p, logs_q)):
        assert {k: v for k, v in lp.items() if not k.startswith("time/") and k not in PAR_KEYS} == \
            {k: v for k, v in lq.items() if not k.startswith("time/")}
        if i % 2 == 0:
            assert PAR_KEYS <= set(lp)
            got, (mean, _, abs_mean, rate) = next(it)
            assert lp["eval/imp_vs_par"] == got["imp_vs_par"][0] == pytest.approx(mean, rel=1e-12, abs=1e-12)
            assert lp["eval/abs_imp_vs_par"] == got["abs_imp_vs_par"] == pytest.approx(abs_mean, rel=1e-12, abs=1e-12)
            assert lp["eval/par_contract_rate"] == got["par_contract_rate"] == pytest.approx(rate, rel=1e-12, abs=1e-12)
        else:
            assert not PAR_KEYS & set(lp)
    pp, pq = params_to_numpy(runner_p[0]), params_to_numpy(runner_q[0])
    assert all((pp[k] == pq[k]).all() for k in pp)


def test_par_imp_training_runs_solo_and_in_a_population(tmp_path):
    from brl_b200 import ppo, random as brandom
    tables, eval_table = _tables()
    _, logs = ppo.train(_train_config(tmp_path, "s", lr=1e-4, reward_mode="par_imp"), brandom.PRNGKey(5), tables=tables,
                        eval_table=eval_table, device=DEV)
    assert len(logs) == 3 and all(np.isfinite(log["train/total_loss"]) and np.isfinite(log["train/value_loss"]) for log in logs)
    modes = ("par_imp", "score", "par_imp")
    out = ppo.train_population([_train_config(tmp_path, f"k{k}", seed=k, lr=1e-4, reward_mode=m) for k, m in enumerate(modes)],
                               [brandom.PRNGKey(10 + k) for k in range(3)], tables=tables, eval_table=eval_table, device=DEV)
    for _, logs in out:
        assert len(logs) == 3 and all(np.isfinite(log["train/total_loss"]) for log in logs)
