"""Population-based training on the GPU (ppo.train_population(..., pbt=...), brl_b200/pbt.py): without a ranking the run is
today's, an exploit step copies the winner's state byte for byte and the loser's next update is the solo update of the
copied state under its perturbed config, the league fitness is the pairwise duplicate matches' mean IMP, and a run that
ranks every iteration keeps its logs and lineage consistent with the copies it made."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _flat(params):
    from brl_b200.models import LAYERS
    return torch.cat([params[name][k].reshape(-1) for name in LAYERS for k in ("w", "b")])


def _bits(t):
    return t.contiguous().view(torch.int32)


def _configs(root, K, iterations):
    base = dict(num_envs=256, num_steps=8, minibatch_size=256, update_epochs=2, total_timesteps=256 * 8 * iterations,
                hash_size=40, num_eval_envs=64, num_prioritized_envs=32, num_eval_step=2, save_model=True, log_path=str(root))
    lrs, ents = (1e-4, 3e-4, 2e-5, 5e-4), (0.001, 0.01, 0.0, 0.005)
    return [dict(base, seed=k, lr=lrs[k], ent_coef=ents[k], exp_name=f"l{k}") for k in range(K)]


def _tables():
    from brl_b200.deals import synthetic_deal_table
    return [synthetic_deal_table(300, seed=k) for k in range(3)], synthetic_deal_table(200, seed=9)


def _rngs(K):
    from brl_b200 import random as brandom
    return [brandom.PRNGKey(10 + k) for k in range(K)]


def _assert_same_run(a, b, what):
    from brl_b200.models import params_to_numpy
    for k, ((runner_a, logs_a), (runner_b, logs_b)) in enumerate(zip(a, b)):
        assert len(logs_a) == len(logs_b)
        for la, lb in zip(logs_a, logs_b):
            keys = sorted(x for x in la if not x.startswith("time/"))
            assert keys == sorted(x for x in lb if not x.startswith("time/")), (what, k)
            for x in keys:
                assert la[x] == lb[x] or (np.isnan(la[x]) and np.isnan(lb[x])), (what, k, x, la[x], lb[x])
        pa, pb = params_to_numpy(runner_a[0]), params_to_numpy(runner_b[0])
        assert all(np.array_equal(pa[x], pb[x]) for x in pa), (what, k)
        assert runner_a[1].count == runner_b[1].count
        assert torch.equal(_bits(runner_a[1].mu), _bits(runner_b[1].mu)) and torch.equal(_bits(runner_a[1].nu), _bits(runner_b[1].nu))


def test_without_a_ranking_the_run_is_unchanged(tmp_path):
    """pbt=None is K independent ppo.train runs (what train_population ran before PBT), bit for bit; so is a PBT run whose
    interval never comes round, though it builds its league"""
    from brl_b200 import ppo
    K, iterations = 3, 3
    tables, eval_table = _tables()
    solo = [ppo.train(c, r, tables=tables, eval_table=eval_table, device=DEV)
            for c, r in zip(_configs(tmp_path / "solo", K, iterations), _rngs(K))]
    plain = ppo.train_population(_configs(tmp_path / "none", K, iterations), _rngs(K), tables=tables, eval_table=eval_table,
                                 device=DEV, pbt=None)
    _assert_same_run(plain, solo, "pbt=None")
    assert not any(os.path.exists(tmp_path / "none" / f"l{k}" / "rl_params" / "pbt_lineage.json") for k in range(K))
    idle = ppo.train_population(_configs(tmp_path / "idle", K, iterations), _rngs(K), tables=tables, eval_table=eval_table,
                                device=DEV, pbt=dict(interval=iterations, metric="league"))
    _assert_same_run(idle, plain, "interval > last iteration")
    for k in range(K):
        with open(tmp_path / "idle" / f"l{k}" / "rl_params" / "pbt_lineage.json") as fh:
            assert json.load(fh) == []


def test_exploit_copies_the_winner_and_the_loser_updates_as_a_solo_run(tmp_path, monkeypatch):
    """forced fitness (learner 1 best, learner 2 worst) at iteration 2 of 4: learner 2 takes learner 1's params, mu, nu
    and count byte for byte, learner 1 is untouched, and learner 2's update at iteration 3 equals make_update_step of the
    copied state under the perturbed config"""
    from brl_b200 import pbt, ppo
    from brl_b200.optim import make_optimizer
    from brl_b200.update import make_update_step
    K, iterations = 3, 4
    keys = ("lr", "ent_coef", "clip_eps", "vf_coef")

    def snap(ln):
        st = ln.runner_state[1]
        return _flat(ln.runner_state[0]).clone(), st.mu.clone(), st.nu.clone(), st.count

    events, calls, fps = [], [], []
    original_exploit = pbt.PopulationBasedTraining.exploit

    def exploit(self, loser, winner, factors):
        before = dict(winner=snap(winner), loser_config=dict(loser.config), winner_config=dict(winner.config))
        original_exploit(self, loser, winner, factors)
        torch.cuda.synchronize()
        events.append(dict(before, loser=loser, factors=factors, loser_after=snap(loser), winner_after=snap(winner)))

    original_make = ppo.make_population_update_step

    def make(configs, fp, optimizers):
        step = original_make(configs, fp, optimizers)
        fps.append(fp)

        def recorded(runner_states, trajs, advs, tgts):
            outs = step(runner_states, trajs, advs, tgts)
            calls.append((runner_states, trajs, advs, tgts, [(_flat(rs[0]).clone(), rs[1].count, rs[1].mu.clone(), rs[1].nu.clone(),
                                                              rs[5], li) for rs, li in outs]))
            return outs
        return recorded

    monkeypatch.setattr(pbt.PopulationBasedTraining, "exploit", exploit)
    monkeypatch.setattr(pbt.PopulationBasedTraining, "fitness", lambda self, learners: np.array([0.0, 1.0, -1.0]))
    monkeypatch.setattr(ppo, "make_population_update_step", make)
    tables, eval_table = _tables()
    seen = [[] for _ in range(K)]
    out = ppo.train_population(_configs(tmp_path, K, iterations), _rngs(K), tables=tables, eval_table=eval_table, device=DEV,
                               log_fns=[s.append for s in seen],
                               pbt=dict(interval=2, metric="score", perturb_keys=keys, perturb_factors=(0.5, 2.0), seed=3))
    assert len(events) == 1 and len(calls) == iterations and len(fps) == 2  # the update step is rebuilt after the step
    ev = events[0]
    # the copy: byte-equal to the winner's state before it; the winner untouched
    for got, want in zip(ev["loser_after"][:3], ev["winner"][:3]):
        assert torch.equal(_bits(got), _bits(want))
    assert ev["loser_after"][3] == ev["winner"][3] == 3 * 2 * 8
    for got, want in zip(ev["winner_after"][:3], ev["winner"][:3]):
        assert torch.equal(_bits(got), _bits(want))
    loser = ev["loser"]
    for key in keys:
        assert loser.config[key] == ev["winner_config"][key] * ev["factors"][key]
        assert ev["factors"][key] in (0.5, 2.0)
    logs = [o[1] for o in out]
    assert [logs[k][2]["pbt/parent"] for k in range(K)] == [-1, -1, 1]
    assert [logs[k][2]["pbt/rank"] for k in range(K)] == [1, 0, 2]
    assert all(logs[2][2][f"pbt/{key}"] == loser.config[key] for key in keys)
    assert seen == logs
    # iteration 3: learner 2's grouped update equals the solo update of its input under the perturbed config
    runner_states, trajs, advs, tgts, results = calls[3]
    rs = runner_states[2]
    assert torch.equal(_bits(_flat(rs[0])), _bits(ev["winner"][0])) and rs[1].count == ev["winner"][3]
    flat_g, count_g, mu_g, nu_g, rng_g, (tl_g, aux_g) = results[2]
    solo = make_update_step(loser.config, fps[1], make_optimizer(loser.config))
    (p_s, st_s, *_, rng_s), (tl_s, aux_s) = solo(rs, trajs[2], advs[2], tgts[2])
    assert torch.equal(_bits(_flat(p_s)), _bits(flat_g)) and st_s.count == count_g == 4 * 2 * 8 and rng_s == rng_g
    assert torch.equal(_bits(st_s.mu), _bits(mu_g)) and torch.equal(_bits(st_s.nu), _bits(nu_g))
    for a, b in zip((tl_s,) + tuple(aux_s), (tl_g,) + tuple(aux_g)):
        assert torch.equal(_bits(a), _bits(b))
    # the config change matters: the same state under the loser's config before the step updates differently
    old = make_update_step(ev["loser_config"], fps[0], make_optimizer(ev["loser_config"]))
    (p_o, *_), _ = old(rs, trajs[2], advs[2], tgts[2])
    assert not torch.equal(_bits(_flat(p_o)), _bits(flat_g))


@pytest.mark.parametrize("K", [3, 4])
def test_league_fitness_is_the_mean_imp_of_the_pairwise_matches(K):
    from brl_b200 import pbt, random as brandom
    from brl_b200.deals import synthetic_deal_table
    from brl_b200.env import BridgeBidding
    from brl_b200.evaluation import make_device_duplicate_evaluate, make_selfplay_league_evaluate
    from brl_b200.models import init_params
    boards = 100
    env = BridgeBidding(table=synthetic_deal_table(200, seed=9), device=DEV)
    nets = [init_params(40 + k, DEV) for k in range(K)]
    key = brandom.PRNGKey(5)
    league = make_selfplay_league_evaluate(env, "relu", "DeepMind", boards)
    returns = {}
    fitness = pbt.league_fitness(league, nets, key, cum_returns=returns)
    again = pbt.league_fitness(league, nets, key)            # the same buffers, relaunched
    assert np.array_equal(fitness, again)
    match = make_device_duplicate_evaluate(env, "relu", "DeepMind", boards)
    imps = np.zeros((K, K))
    for i in range(K):
        for j in range(i + 1, K):
            log_info, _, _, cum_return = match(nets[i], nets[j], key)
            assert torch.equal(_bits(cum_return), _bits(returns[(i, j)])), (i, j)
            imps[i, j], imps[j, i] = log_info[0], -log_info[0]
    want = np.array([sum(imps[k, j] for j in range(K) if j != k) / (K - 1) for k in range(K)])
    np.testing.assert_allclose(fitness, want, rtol=1e-12, atol=1e-12)
    assert len(set(np.round(fitness, 9))) > 1                 # the nets play differently: a real ranking


@pytest.mark.parametrize("metric", ["league", "score"])
def test_a_population_that_ranks_every_iteration(tmp_path, metric):
    """K = 4, interval = 1, 3 iterations: rankings at iterations 1 and 2, one loser each (n = 1); the pbt/* logs, the
    learners' lr schedule and the lineage files agree with the copies, and the last copy leaves the loser's final state
    equal to its parent's"""
    from brl_b200 import ppo
    K, iterations, keys = 4, 3, ("lr", "ent_coef")
    tables, eval_table = _tables()
    seen = [[] for _ in range(K)]
    configs = _configs(tmp_path, K, iterations)
    out = ppo.train_population(configs, _rngs(K), tables=tables, eval_table=eval_table, device=DEV,
                               log_fns=[(lambda log, s=s: s.append(dict(log))) for s in seen],
                               pbt=dict(interval=1, metric=metric, seed=1))
    logs = [o[1] for o in out]
    assert all(len(lg) == iterations for lg in logs)
    assert not any(x.startswith("pbt/") for lg in logs for x in lg[0])
    values = [{key: configs[k][key] for key in keys} for k in range(K)]
    for i in (1, 2):
        at = [logs[k][i] for k in range(K)]
        assert all(all(x in seen[k][i] for x in at[k] if x.startswith("pbt/")) for k in range(K))  # logged before log_fn
        fit = [a["pbt/fitness"] for a in at]
        if metric == "score":
            assert fit == [a["train/score"] for a in at]
        order = sorted(range(K), key=lambda k: (-fit[k], k))
        assert [at[k]["pbt/rank"] for k in range(K)] == [order.index(k) for k in range(K)]
        parents = [a["pbt/parent"] for a in at]
        loser = order[-1]
        assert parents == [order[0] if k == loser else -1 for k in range(K)]
        for k in range(K):
            for key in keys:
                if k == loser:  # the parent's value times one of the factors
                    assert any(at[k][f"pbt/{key}"] == values[order[0]][key] * f for f in (0.8, 1.25)), (i, key)
                else:
                    assert at[k][f"pbt/{key}"] == values[k][key], (i, k, key)
        values = [{key: at[k][f"pbt/{key}"] for key in keys} for k in range(K)]
        if i == 1:  # the next iteration steps with the new learning rates (no annealing)
            assert [logs[k][2]["train/lr"] for k in range(K)] == [values[k]["lr"] for k in range(K)]
    # lineage files: one entry per ranking
    for k in range(K):
        with open(tmp_path / f"l{k}" / "rl_params" / "pbt_lineage.json") as fh:
            lineage = json.load(fh)
        assert lineage == [[i, logs[k][i]["pbt/parent"], {key: logs[k][i][f"pbt/{key}"] for key in keys}] for i in (1, 2)]
    # the last ranking is after the last update: the loser ends with its parent's state
    loser = next(k for k in range(K) if logs[k][2]["pbt/parent"] != -1)
    parent = logs[loser][2]["pbt/parent"]
    (p_l, st_l, *_), (p_p, st_p, *_) = out[loser][0], out[parent][0]
    assert torch.equal(_bits(_flat(p_l)), _bits(_flat(p_p))) and st_l.count == st_p.count
    assert torch.equal(_bits(st_l.mu), _bits(st_p.mu)) and torch.equal(_bits(st_l.nu), _bits(st_p.nu))
