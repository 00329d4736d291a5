"""Population-based training without a GPU: the ranking, selection and perturbation decisions from given fitness vectors,
the option checks of train_population's `pbt` (which run before any device work) and the lineage file's layout."""
import json
import math
from fractions import Fraction

import numpy as np
import pytest


def _config(**kw):
    c = dict(num_envs=64, num_steps=4, minibatch_size=64, update_epochs=2, total_timesteps=4096, lr=1e-3, ent_coef=0.01,
             seed=0)
    c.update(kw)
    return c


def _plan(fitness, quantile=0.25, keys=("lr", "ent_coef"), factors=(0.8, 1.25), seed=0):
    from brl_b200 import pbt
    return pbt.plan(fitness, quantile, keys, factors, np.random.default_rng(seed))


def test_default_pbt_config():
    from brl_b200 import ppo
    assert ppo.default_pbt_config() == dict(interval=10, metric="league", league_boards=100, quantile=0.25,
                                            perturb_keys=("lr", "ent_coef"), perturb_factors=(0.8, 1.25), seed=0)


@pytest.mark.parametrize("quantile", ["1/20", "1/10", "1/4", "3/10", "1/3", "1/2"])
def test_n_for_every_population_size(quantile):
    """n = max(1, floor(quantile * K)) in exact arithmetic, for the float quantile a user passes"""
    from brl_b200 import pbt
    q = Fraction(quantile)
    for K in range(2, 65):
        n = pbt.num_exploit(K, float(q))
        assert n == max(1, math.floor(q * K)), (K, quantile)
        assert 1 <= n <= K // 2  # the bottom and top sets never overlap
        ranks, moves = _plan(np.arange(K, dtype=np.float64), float(q))
        assert len(moves) == n and sorted(ranks) == list(range(K))


def test_bottom_losers_copy_top_winners():
    fitness = np.array([0.5, -2.0, 3.0, 1.0, -1.0, 2.5, 0.0, -3.0])   # order: 2, 5, 3, 0, 6, 4, 1, 7
    ranks, moves = _plan(fitness, quantile=0.25)                        # n = 2
    assert ranks == [3, 6, 0, 2, 5, 1, 4, 7]
    assert [m[0] for m in moves] == [1, 7]                               # the two lowest, in index order
    assert all(w in (2, 5) for _, w, _ in moves)
    for _, _, f in moves:
        assert sorted(f) == ["ent_coef", "lr"] and all(v in (0.8, 1.25) for v in f.values())


def test_ties_go_to_the_lower_index():
    from brl_b200 import pbt
    assert pbt.rank_order([1.0, 1.0, 1.0, 1.0]) == [0, 1, 2, 3]
    ranks, moves = _plan([1.0, 1.0, 1.0, 1.0], quantile=0.25)
    assert ranks == [0, 1, 2, 3] and [(m[0], m[1]) for m in moves] == [(3, 0)]
    ranks, moves = _plan([2.0, 5.0, 2.0, 5.0, 2.0, 2.0], quantile=0.5)   # n = 3
    assert ranks == [2, 0, 3, 1, 4, 5]
    assert [m[0] for m in moves] == [2, 4, 5] and all(m[1] in (1, 3, 0) for m in moves)
    # a NaN fitness (a diverged learner) ranks last
    assert pbt.rank_order([0.0, math.nan, -1.0]) == [0, 2, 1]


def test_the_plan_is_deterministic_under_its_seed():
    rng = np.random.default_rng(3)
    fitness = rng.normal(size=16)
    a = [_plan(fitness, seed=7) for _ in range(2)]
    assert a[0] == a[1]
    plans = {str(_plan(fitness, seed=s)[1]) for s in range(20)}
    assert len(plans) > 1                                                # the seed drives winners and factors
    # successive steps draw from one generator in a fixed order: winner, then one factor per key, loser by loser
    from brl_b200 import pbt
    g, h = np.random.default_rng(11), np.random.default_rng(11)
    for step in range(3):
        _, moves = pbt.plan(fitness + step, 0.25, ("lr", "ent_coef"), (0.8, 1.25), g)
        top = pbt.rank_order(fitness + step)[:4]
        for loser, winner, factors in moves:
            assert winner == top[int(h.integers(4))]
            assert factors == {"lr": (0.8, 1.25)[int(h.integers(2))], "ent_coef": (0.8, 1.25)[int(h.integers(2))]}


def test_factor_application():
    from brl_b200 import pbt
    got = pbt.explore({"lr": 3e-4, "ent_coef": 0.01, "vf_coef": 0.5}, {"lr": 1.25, "ent_coef": 0.8})
    assert got == {"lr": 3e-4 * 1.25, "ent_coef": 0.01 * 0.8}
    assert pbt.explore({"lr": 1e-3}, {}) == {}
    ranks, moves = _plan([0.0, 1.0, 2.0, 3.0], keys=("clip_eps",), factors=(2.0,))
    assert moves == [(0, 3, {"clip_eps": 2.0})]


@pytest.mark.parametrize("pbt,match", [
    (dict(perturb_keys=("num_envs",)), "num_envs"),                 # shared by the population
    (dict(perturb_keys=("minibatch_size", "lr")), "minibatch_size"),
    (dict(perturb_keys=("lr", "learning_rate")), "learning_rate"),  # unknown to default_config()
    (dict(perturb_keys=("seed",)), "seed"),                         # a config key, but no hyperparameter to scale
    (dict(quantile=0.0), "quantile"),
    (dict(quantile=0.51), "quantile"),
    (dict(quantile=-0.25), "quantile"),
    (dict(interval=0), "interval"),
    (dict(league_boards=0), "league_boards"),
    (dict(metric="elo"), "metric"),
    (dict(perturb_factors=()), "perturb_factors"),
    (dict(perturb_factors=(0.8, -1.0)), "perturb_factors"),
    (dict(intervall=5), "intervall"),
])
def test_bad_pbt_options_are_refused_before_any_device_work(pbt, match):
    from brl_b200 import ppo
    with pytest.raises(ValueError, match=match):
        ppo.train_population([_config(), _config(seed=1)], [0, 1], device="cpu", pbt=pbt)


def test_pbt_needs_two_learners():
    from brl_b200 import ppo
    with pytest.raises(ValueError, match="at least 2"):
        ppo.train_population([_config()], [0], device="cpu", pbt={})


def test_good_pbt_options():
    from brl_b200 import pbt
    cfg = pbt.check_pbt_config(dict(quantile=0.5, perturb_keys="lr", perturb_factors=[0.5, 2], interval=1), 2)
    assert cfg["perturb_keys"] == ("lr",) and cfg["perturb_factors"] == (0.5, 2.0) and cfg["metric"] == "league"
    for key in pbt.PERTURBABLE_KEYS:
        pbt.check_pbt_config(dict(perturb_keys=(key,)), 3)


def test_lineage_file_layout(tmp_path):
    from brl_b200 import pbt
    path = tmp_path / "pbt_lineage.json"
    pbt.write_lineage(str(path), [[10, -1, {"lr": 1e-6, "ent_coef": 0.001}], [20, np.int64(3), {"lr": np.float64(1.25e-6),
                                                                                                   "ent_coef": 0.0008}]])
    assert json.loads(path.read_text()) == [[10, -1, {"lr": 1e-6, "ent_coef": 0.001}], [20, 3, {"lr": 1.25e-6, "ent_coef": 0.0008}]]
