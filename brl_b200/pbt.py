"""Population-based training (PBT; Jaderberg et al. 2017, "Population Based Training of Neural Networks") for
`ppo.train_population`.

Every `interval` iterations the K learners are ranked.  Each of the n = max(1, floor(quantile * K)) lowest takes the
parameters and Adam state of one of the n highest ("exploit") and continues with that learner's hyperparameters, each of
`perturb_keys` multiplied by a factor drawn from `perturb_factors` ("explore").  The loser keeps everything else of its
own: env state, rollout key, deal-table rotation, opponent zoo and save directory.

The ranking ("metric") is either a round-robin league of the K current nets -- one `make_selfplay_league_evaluate` call,
every pair playing a duplicate match on the same `league_boards` boards of the eval table, fitness = a learner's mean IMP
over its K - 1 matches -- or each learner's latest `train/score`.  Ties go to the lower learner index.  Which loser copies
which winner, and the factors, come from one `np.random.Generator(seed)` of the population, so a run is deterministic and
the learners' own generators (opponent and zoo draws) are not touched.  The copies are device-to-device `copy_` calls on
the current stream; the only host read of a PBT step is the league's statistics."""
from __future__ import annotations

import json
import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

# The hyperparameters an explore step may multiply: the loss coefficients (the KL anchor's among them) and the optimizer's
# (read by the update step and the optimizer, rebuilt after each change) and GAE's (read by calc_gae at every call).  Keys
# of update.POPULATION_SHARED_KEYS fix shapes or launch flags and cannot differ between learners.  A loser keeps its own
# anchor net and takes the winner's anchor_kl_coef times the factor.
PERTURBABLE_KEYS = ("lr", "ent_coef", "vf_coef", "clip_eps", "max_grad_norm", "illegal_action_l2norm_coef", "gamma",
                    "gae_lambda", "anchor_kl_coef")

METRICS = ("league", "score")


def default_pbt_config() -> dict:
    """The PBT options of `ppo.train_population(..., pbt=...)` and their defaults."""
    return dict(interval=10, metric="league", league_boards=100, quantile=0.25, perturb_keys=("lr", "ent_coef"),
                perturb_factors=(0.8, 1.25), seed=0)


def check_pbt_config(pbt: dict, num_learners: int) -> dict:
    """default_pbt_config() updated with `pbt`, checked: ValueError for an unknown option, a population of fewer than two
    learners, an interval or board count below 1, an unknown metric, a quantile outside (0, 0.5], a perturbed key that
    default_config() does not know, that the population shares (update.POPULATION_SHARED_KEYS) or that is not one of
    PERTURBABLE_KEYS, and a factor that is not a finite positive number."""
    from .ppo import default_config
    from .update import POPULATION_SHARED_KEYS
    cfg = default_pbt_config()
    unknown = sorted(set(pbt) - set(cfg))
    if unknown:
        raise ValueError(f"unknown PBT option(s) {unknown}; the options are {sorted(cfg)}")
    cfg.update(pbt)
    if num_learners < 2:
        raise ValueError(f"PBT needs a population of at least 2 learners; got {num_learners}")
    for key in ("interval", "league_boards"):
        if isinstance(cfg[key], bool) or not isinstance(cfg[key], (int, np.integer)) or cfg[key] < 1:
            raise ValueError(f"PBT option {key!r} must be an integer >= 1; got {cfg[key]!r}")
    if cfg["metric"] not in METRICS:
        raise ValueError(f"PBT metric must be one of {METRICS}; got {cfg['metric']!r}")
    q = cfg["quantile"]
    if not (isinstance(q, (int, float)) and 0.0 < q <= 0.5):
        raise ValueError(f"PBT quantile must lie in (0, 0.5]; got {q!r}")
    keys = cfg["perturb_keys"]
    keys = (keys,) if isinstance(keys, str) else tuple(keys)
    known = default_config()
    for key in keys:
        if key not in known:
            raise ValueError(f"PBT perturb key {key!r} is not a config key (default_config())")
        if key in POPULATION_SHARED_KEYS:
            raise ValueError(f"PBT perturb key {key!r} must be equal across the population (update.POPULATION_SHARED_KEYS)")
        if key not in PERTURBABLE_KEYS:
            raise ValueError(f"PBT perturb key {key!r} is not a hyperparameter PBT can perturb {PERTURBABLE_KEYS}")
    factors = tuple(float(f) for f in cfg["perturb_factors"])
    if not factors or not all(math.isfinite(f) and f > 0.0 for f in factors):
        raise ValueError(f"PBT perturb_factors must be finite positive numbers; got {cfg['perturb_factors']!r}")
    cfg["perturb_keys"], cfg["perturb_factors"] = keys, factors
    cfg["seed"] = int(cfg["seed"])
    return cfg


def num_exploit(num_learners: int, quantile: float) -> int:
    """n = max(1, floor(quantile * K)): the size of the bottom set that is replaced and of the top set it draws from"""
    return max(1, int(math.floor(quantile * num_learners + 1e-9)))


def rank_order(fitness: Sequence[float]) -> List[int]:
    """learner indices from the fittest down; ties go to the lower index, a NaN fitness ranks last"""
    f = [-math.inf if math.isnan(x) else float(x) for x in fitness]
    return sorted(range(len(f)), key=lambda k: (-f[k], k))


def plan(fitness: Sequence[float], quantile: float, perturb_keys: Sequence[str], perturb_factors: Sequence[float],
         gen: np.random.Generator) -> Tuple[List[int], List[Tuple[int, int, Dict[str, float]]]]:
    """One PBT step's decisions from the fitness vector -> (ranks, moves).  ranks[k] is learner k's place (0 = fittest).
    moves holds, for each of the n lowest learners in index order, (loser, winner, {key: factor}): the winner drawn
    uniformly from the n highest, then one factor per perturbed key, all from `gen` in that order."""
    order = rank_order(fitness)
    K = len(order)
    n = num_exploit(K, quantile)
    ranks = [0] * K
    for r, k in enumerate(order):
        ranks[k] = r
    top, bottom = order[:n], sorted(order[K - n:])
    moves = []
    for loser in bottom:
        winner = top[int(gen.integers(n))]
        factors = {key: float(perturb_factors[int(gen.integers(len(perturb_factors)))]) for key in perturb_keys}
        moves.append((loser, winner, factors))
    return ranks, moves


def explore(values: Dict[str, float], factors: Dict[str, float]) -> Dict[str, float]:
    """the winner's hyperparameter values, each multiplied by its factor"""
    return {key: float(values[key]) * factors[key] for key in factors}


def league_fitness(league, params_list, rng_key, cum_returns: Optional[dict] = None) -> np.ndarray:
    """One `make_selfplay_league_evaluate` call over the nets of `params_list` -> float64[K]: net k's mean IMP over its
    K - 1 matches (column k of league_matrices' win_lose holds k's IMP against each other net).  `cum_returns` (a dict)
    receives each pair's per-env returns."""
    _, win_lose, _, _ = league(params_list, rng_key, cum_returns=cum_returns)
    return win_lose.sum(axis=0) / (len(params_list) - 1)


def write_lineage(path: str, lineage) -> None:
    """pbt_lineage.json: one [iteration, parent, {key: value}] per PBT step -- the learner it copied (-1: none) and its
    perturbed hyperparameters after the step"""
    with open(path, "w") as fh:
        json.dump([[int(i), int(parent), {k: float(v) for k, v in values.items()}] for i, parent, values in lineage], fh)


class PopulationBasedTraining:
    """The PBT control plane of one population: `due(i)` says whether iteration i ranks (i > 0 and i % interval == 0),
    `step(i, learners)` ranks, exploits and explores after every learner's finish_iteration, adds the pbt/* entries to
    each learner's latest log and its lineage.  Every step replaces at least one learner's config, so the caller then
    rebuilds the population update step, which holds the loss coefficients and the optimizers."""

    def __init__(self, cfg: dict, learners):
        self.cfg = cfg
        self.gen = np.random.default_rng(cfg["seed"])
        self.league = None
        if cfg["metric"] == "league":  # built once: its pool and match buffers are allocated at the first ranking
            from .evaluation import make_selfplay_league_evaluate
            c = learners[0].config
            self.league = make_selfplay_league_evaluate(learners[0].eval_env, c["actor_activation"], c["actor_model_type"],
                                                        cfg["league_boards"])
        for ln in learners:
            ln.pbt_lineage = []

    def due(self, i: int) -> bool:
        return i > 0 and i % self.cfg["interval"] == 0

    def fitness(self, learners) -> np.ndarray:
        """"league": the K current nets' round robin on the eval table, keyed by learner 0's evaluation key (every learner
        evaluates on the same table); "score": each learner's latest train/score"""
        if self.league is None:
            return np.array([ln.logs[-1]["train/score"] for ln in learners], dtype=np.float64)
        return league_fitness(self.league, [ln.runner_state[0] for ln in learners], learners[0].eval_rng)

    def exploit(self, loser, winner, factors: Dict[str, float]) -> None:
        loser.adopt(winner, explore({key: winner.config[key] for key in factors}, factors))

    def step(self, i: int, learners) -> None:
        cfg = self.cfg
        fit = self.fitness(learners)
        ranks, moves = plan(fit, cfg["quantile"], cfg["perturb_keys"], cfg["perturb_factors"], self.gen)
        parents = [-1] * len(learners)
        for loser, winner, factors in moves:
            self.exploit(learners[loser], learners[winner], factors)
            parents[loser] = winner
        for k, ln in enumerate(learners):
            values = {key: float(ln.config[key]) for key in cfg["perturb_keys"]}
            ln.logs[-1].update({"pbt/fitness": float(fit[k]), "pbt/rank": ranks[k], "pbt/parent": parents[k]})
            ln.logs[-1].update({f"pbt/{key}": v for key, v in values.items()})
            ln.pbt_lineage.append([i, parents[k], values])
