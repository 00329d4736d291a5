"""CPU: partnerships of two different nets (DESIGN.md f14) -- the NumPy restatement of brl_model_rows by player id, the pair
layout of cross-play, the fixed-partner config rules of ppo.train / train_population, PBT's adopt keeping a learner's
partner, and the argument checks of BRL_F_PLAYER_MODELS and BRL_F_EVAL_PARTNER."""
import ctypes
import pickle

import numpy as np
import pytest
import torch


def ref_player_grouping(player, done, env_models, M, rows_per_group=256):
    """brl_model_rows restated: the acting net of each live env (env_models[i, player] for [n, 4], [i, player >= 2] for
    [n, 2]); -> (counts[M], offsets[M + 1] padded to 256-row groups with offsets[M] = -1 on a live out-of-range id, each
    group's sorted env ids, the group id of every 256-row block)"""
    n = player.shape[0]
    col = (player & 3) if env_models.shape[1] == 4 else (player >= 2).astype(np.int64)
    acting = env_models[np.arange(n), col] if n else np.zeros(0, np.int32)
    live = done == 0
    bad = bool((live & ((acting < 0) | (acting >= M))).any())
    counts = np.array([int((live & (acting == m)).sum()) for m in range(M)], dtype=np.int32)
    padded = (counts + rows_per_group - 1) // rows_per_group * rows_per_group
    offsets = np.concatenate([[0], np.cumsum(padded)]).astype(np.int32)
    blocks = np.concatenate([np.full(p // rows_per_group, m, np.int32) for m, p in enumerate(padded)] + [np.zeros(0, np.int32)])
    rows = [sorted(np.flatnonzero(live & (acting == m)).tolist()) for m in range(M)]
    if bad:
        offsets[M] = -1
    return counts, offsets, rows, blocks


def test_the_restatement_on_a_hand_made_batch():
    player = np.array([0, 1, 2, 3, 1, 0], np.int8)
    done = np.array([0, 0, 0, 0, 1, 0], np.uint8)
    ids = np.array([[0, 1, 2, 2], [0, 1, 2, 2], [0, 1, 2, 1], [0, 1, 2, 1], [0, 1, 2, 2], [1, 0, 2, 2]], np.int32)
    counts, offsets, rows, blocks = ref_player_grouping(player, done, ids, 3)
    # env 3 acts for player 3, whose net is env_models[3, 3] = 1; env 4 is finished and not listed
    assert counts.tolist() == [1, 3, 1] and offsets.tolist() == [0, 256, 512, 768] and blocks.tolist() == [0, 1, 2]
    assert rows == [[0], [1, 3, 5], [2]]
    # partners on one net: the by-player grouping is the by-team one
    team = ids[:, [0, 2]]
    same = team[:, [0, 0, 1, 1]]
    for a, b in zip(ref_player_grouping(player, done, same, 3), ref_player_grouping(player, done, team, 3)):
        assert (np.asarray(a, dtype=object) == np.asarray(b, dtype=object)).all()
    bad = ids.copy()
    bad[2, 2] = 3
    assert ref_player_grouping(player, done, bad, 3)[1][3] == -1
    bad[2, 2], done[2] = 3, 1   # an out-of-range id on a finished env is never read
    assert ref_player_grouping(player, done, bad, 3)[1][3] == 512


@pytest.mark.parametrize("M,n,per_chunk,world", [(1, 100, 1, 1), (3, 100, 2, 2), (8, 100, 10, 3), (16, 100, 7, 8)])
def test_pair_chunk_layout_over_the_partnerships(M, n, per_chunk, world):
    """cross-play's M^2 matches (a, b, c, d) in (a, b) row-major order: every board of every match is played exactly once,
    by the rank and chunk the layout assigns, whatever the rank count"""
    from brl_b200.evaluation import pair_chunk_layout
    pairs = [(a, b, M, M + 1) for a in range(M) for b in range(M)]
    seen = np.zeros((len(pairs), n), dtype=np.int64)
    for rank in range(world):
        for c0, P, lo, hi, p_lo, p_hi, bounds in pair_chunk_layout(len(pairs), n, per_chunk, rank, world):
            g = np.arange(lo, hi)
            arr = np.asarray(pairs, dtype=np.int32).reshape(-1, 4)[c0 + g // n]
            assert arr.shape == (hi - lo, 4) and (arr[:, 2] == M).all() and (arr[:, 3] == M + 1).all()
            np.add.at(seen, (c0 + g // n, g % n), 1)
            for p in range(p_lo, p_hi):
                assert bounds[p - p_lo + 1] - bounds[p - p_lo] == ((c0 + g // n) == c0 + p).sum()
    assert (seen == 1).all()


def _save(path, params):
    with open(path, "wb") as fh:
        pickle.dump(params, fh)
    return str(path)


def _net(shapes=None):
    from brl_b200.models import LAYERS, SIZES
    shapes = shapes or {}
    return {name: {"w": np.zeros(shapes.get(name, (fi, fo)), np.float32), "b": np.zeros(fo, np.float32)}
            for name, (fi, fo) in zip(LAYERS, SIZES)}


def test_partner_config_rules(tmp_path):
    from brl_b200 import ppo
    from brl_b200.models import LAYERS
    good = _save(tmp_path / "good.pkl", _net())
    assert ppo.default_config()["partner_model_path"] is None
    ppo.check_partner_config(ppo.default_config())
    ppo.check_partner_config(dict(ppo.default_config(), partner_model_path=good))
    wide = _save(tmp_path / "wide.pkl", _net({LAYERS[1]: (1024, 512)}))
    short = _save(tmp_path / "short.pkl", {k: v for k, v in _net().items() if k != LAYERS[5]})
    for kw, match in ((dict(partner_model_path=good, ratio_model_zoo=0.5), "ratio_model_zoo"),
                      (dict(partner_model_path=wide), "DeepMind 4x1024"),
                      (dict(partner_model_path=short), "DeepMind 4x1024")):
        with pytest.raises(ValueError, match=match):
            ppo.check_partner_config(dict(ppo.default_config(), **kw))
        with pytest.raises(ValueError, match=match):   # before any device work: no device is touched on this CPU machine
            ppo.train(kw, 0, device="cpu")
        with pytest.raises(ValueError, match=match):
            ppo.train_population([{}, kw], [0, 1], device="cpu")


def test_a_population_may_mix_partnered_and_unpartnered_learners(tmp_path):
    from brl_b200 import ppo
    from brl_b200.pbt import check_pbt_config
    from brl_b200.update import check_population_configs
    good = _save(tmp_path / "good.pkl", _net())
    configs = [ppo.full_config(dict(partner_model_path=good)), ppo.full_config({}), ppo.full_config(dict(partner_model_path=good))]
    check_population_configs(configs)
    for c in configs:
        ppo.check_partner_config(c)
    with pytest.raises(ValueError, match="partner_model_path"):
        check_pbt_config(dict(perturb_keys=("lr", "partner_model_path")), 4)


def test_pbt_adopt_keeps_the_losers_partner():
    from brl_b200 import ppo
    from brl_b200.models import LAYERS
    from brl_b200.optim import OptState

    def learner(value, partner):
        ln = ppo.Learner.__new__(ppo.Learner)
        params = {name: {k: torch.full((3,), float(value)) for k in ("w", "b")} for name in LAYERS}
        ln.runner_state = (params, OptState(value, torch.full((4,), float(value)), torch.full((4,), float(value))), "env", "obs",
                           0, value)
        ln.config = ppo.full_config(dict(lr=1e-4 * value, self_play=True))
        ln.partner_params = partner
        return ln
    winner, loser = learner(1, {"net": "winner's partner"}), learner(2, {"net": "loser's partner"})
    keep = loser.partner_params
    loser.adopt(winner, {"lr": 3e-4})
    assert loser.partner_params is keep and winner.partner_params["net"] == "winner's partner"
    assert torch.equal(loser.runner_state[0][LAYERS[0]]["w"], winner.runner_state[0][LAYERS[0]]["w"])
    assert loser.config["lr"] == 3e-4 and loser.opp_params is loser.runner_state[0]


def _bind(L, name):
    fn = getattr(L, name)
    fn.restype, fn.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]
    return fn


def test_new_flags_are_checked_without_a_gpu():
    from brl_b200 import _lib, ops
    L = _lib.load()
    assert L.brl_xla_layout(b"brl_duplicate_match") == b"iiiiisoxooooooooooooo"   # flags only: the layouts are unchanged
    assert L.brl_xla_layout(b"brl_evaluate_match") == b"iiisoox" + b"o" * 19
    assert "brl_evaluate_match_partner_scratch_bytes" in _lib.MISC
    assert _lib.F_PLAYER_MODELS & _lib.F_EVAL_PARTNER == 0
    # brl_duplicate_match: BRL_F_PLAYER_MODELS needs env_models [3]
    dup = _bind(L, "brl_duplicate_match")
    fake = [4096] * 3 + [None, None, 4096, 4096, 4096, 4096] + [None] * 12
    p = _lib.BrlParams(100, 0, 0, 0, 100, _lib.F_PLAYER_MODELS, 0, 3, -1.0, 1.0, 0.0, 0.0)
    assert dup(None, (ctypes.c_void_p * 21)(*fake), ctypes.byref(p), ctypes.sizeof(p)) == -2
    assert b"BRL_F_PLAYER_MODELS" in L.brl_last_error()
    p.flags = 0  # without the flag a NULL env_models means the default 2-net match: M = 3 is the error
    assert dup(None, (ctypes.c_void_p * 21)(*fake), ctypes.byref(p), ctypes.sizeof(p)) == -1
    # brl_evaluate_match: BRL_F_EVAL_PARTNER needs k_steps = 3
    ev = _bind(L, "brl_evaluate_match")
    fake = [4096] * 8 + [None] * 18
    for k_steps in (0, 2, 4):
        p = _lib.BrlParams(100, 0, 0, 0, 100, _lib.f_eval_match(_lib.EVAL_MATCH_DUPLICATE) | _lib.F_EVAL_PARTNER, 0, k_steps,
                           -1.0, 1.0, 0.0, 0.0)
        assert ev(None, (ctypes.c_void_p * 26)(*fake), ctypes.byref(p), ctypes.sizeof(p)) == -1
        assert b"BRL_F_EVAL_PARTNER" in L.brl_last_error()
    # the partner's scratch holds a third net and nets by player id
    for mode in (_lib.EVAL_MATCH_DUPLICATE, _lib.EVAL_MATCH_SINGLE, _lib.EVAL_MATCH_SIMPLE):
        assert ops.evaluate_match_scratch_bytes(0, mode, partner=True) == 0
        for n in (1, 1000, 4097):
            plain, partner = ops.evaluate_match_scratch_bytes(n, mode), ops.evaluate_match_scratch_bytes(n, mode, partner=True)
            assert partner % 256 == 0 and (partner > plain if n > 1 else partner >= plain)
    assert ops.evaluate_match_scratch_bytes(100, 4, partner=True) == 0
    # the Python wrappers: shapes of env_models and of the partner's pool
    keys, table = torch.zeros(10, dtype=torch.int64), torch.zeros((100, 48), dtype=torch.uint8)
    pool2 = torch.zeros((2, ops.mlp_pool_stride()), dtype=torch.uint8)
    cum, status = torch.zeros(10), torch.zeros(1, dtype=torch.int32)
    acc, sums = torch.zeros((10, _lib.EVAL_ACC_COLS)), torch.zeros(L.brl_eval_num_sums(), dtype=torch.float64)
    scratch = torch.zeros(ops.evaluate_match_scratch_bytes(10, 1, partner=True), dtype=torch.uint8)
    with pytest.raises(_lib.BrlError, match=r"u8\[3, mlp_pool_stride\(\)\]"):
        ops.evaluate_match(keys, table, pool2, scratch, cum, status, mode=1, acc=acc, sums=sums, partner=True)
    with pytest.raises(_lib.BrlError, match=r"\[n, 4\]"):
        ops.duplicate_match(keys, table, torch.zeros((3, ops.mlp_pool_stride()), dtype=torch.uint8), scratch, cum,
                            torch.zeros(8, dtype=torch.float64), status, env_models=torch.zeros((10, 3), dtype=torch.int32))
    rows = torch.zeros(ops.model_rows_capacity(10, 3), dtype=torch.int32)
    with pytest.raises(_lib.BrlError, match=r"\[n, 4\]"):
        ops.model_rows(torch.zeros(10, dtype=torch.int8), None, torch.zeros((10, 3), dtype=torch.int32), rows,
                       torch.zeros(3, dtype=torch.int32), torch.zeros(4, dtype=torch.int32), torch.zeros(8, dtype=torch.int32))


def test_host_scripts_parse_their_arguments():
    import importlib
    crossplay = importlib.import_module("scripts.crossplay")
    cfg = crossplay.parse_args(["exp_name=run", "opp_model_path=sl.pkl", "num_eval_envs=64"])
    assert cfg["exp_name"] == "run" and cfg["num_eval_envs"] == 64 and cfg["partner_opp_model_path"] == ""
    with pytest.raises(SystemExit):
        crossplay.parse_args(["exp_name=run"])
    with pytest.raises(SystemExit):
        crossplay.parse_args(["nope=1", "opp_model_path=x"])
