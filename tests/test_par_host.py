"""CPU: the double-dummy par reference (tests/par_ref.py) on boards worked by hand and on its properties, the reward-mode
config checks, and the argument checks of brl_par / brl_gather_reward_par / brl_par_stats (no device needed)."""
import ctypes

import numpy as np
import pytest

from tests import helpers as H
from tests import par_ref as P


def _sacrifice_board():
    """NS make exactly 10 tricks in spades, EW 9 in hearts; every other strain 6 tricks for everyone"""
    dd = np.full((4, 5), 6, dtype=np.int32)
    dd[0, 3] = dd[2, 3] = 10
    dd[1, 2] = dd[3, 2] = 9
    return dd


def test_sacrifice_over_a_game_is_par_when_the_sacrificers_are_not_vulnerable():
    v, contract = P.par(_sacrifice_board(), dealer=0, vul_ns=0, vul_ew=0)
    assert v == 300                                     # 5Hx by EW down 2 (not vulnerable) beats 4S by NS (+420)
    assert contract == 22 | 1 << 8 | 1 << 10           # 5H, E declares (E and W tie: E comes first after dealer N), doubled


def test_game_is_par_when_the_sacrifice_costs_more():
    v, contract = P.par(_sacrifice_board(), dealer=0, vul_ns=0, vul_ew=1)
    assert (v, contract) == (420, 18)                  # 5Hx would cost 500 vulnerable: 4S by N, +420


def test_no_side_takes_seven_tricks_passes_the_board_out():
    dd = np.full((4, 5), 6, dtype=np.int32)
    for dealer in range(4):
        for vns in (0, 1):
            for vew in (0, 1):
                assert P.par(dd, dealer, vns, vew) == (0, P.PASSED_OUT)


def test_par_depends_on_the_dealer():
    """every seat takes exactly 7 tricks in NT and 6 in each suit: the dealer's side opens 1NT and the other side cannot
    compete profitably"""
    dd = np.full((4, 5), 6, dtype=np.int32)
    dd[:, 4] = 7
    for dealer in range(4):
        v, contract = P.par(dd, dealer, 0, 0)
        assert v == (90 if dealer % 2 == 0 else -90)
        assert contract == 4 | dealer << 8              # 1NT by the dealer (all tie: the dealer comes first), undoubled


def _random_boards(n, seed):
    rng = np.random.default_rng(seed)
    b = H.load_boards()
    from brl_b200.deals import unpack_deal_table
    dd = unpack_deal_table(b["table"])[1]
    idx = rng.integers(0, len(dd), n)
    return dd[idx], rng.integers(0, 4, n), rng.integers(0, 2, n), rng.integers(0, 2, n)


def test_par_is_seating_invariant_and_in_the_rewards_layout():
    dd, dealer, vns, vew = _random_boards(40, 1)
    for k in range(len(dd)):
        v, _ = P.par(dd[k], dealer[k], vns[k], vew[k])
        layouts = [P.par_by_player(v, s) for s in H.SEATINGS]
        for s, lay in zip(H.SEATINGS, layouts):
            assert lay[0] == lay[1] == -lay[2] == -lay[3]
            team_ns = np.array([lay[p] for p in s[[0, 2]]])  # the players seated N and S get the NS par
            assert (team_ns == v).all()


def test_playing_the_par_contract_scores_zero_imps_against_par():
    """a table whose final contract is the par contract, doubled exactly when it fails, scores par"""
    dd, dealer, vns, vew = _random_boards(200, 2)
    n_contracts = 0
    for k in range(len(dd)):
        v, contract = P.par(dd[k], dealer[k], vns[k], vew[k])
        if contract == P.PASSED_OUT:
            score_ns = 0
        else:
            bid, seat, doubled = contract & 0xFF, (contract >> 8) & 3, (contract >> 10) & 1
            t = dd[k][seat][bid % 5]
            assert doubled == (t < bid // 5 + 7)
            s = P.contract_score(bid, doubled, (vns[k], vew[k])[seat % 2], t)
            score_ns = s if seat % 2 == 0 else -s
            n_contracts += 1
        assert P.imp(score_ns - v) == 0
    assert n_contracts > 100


def test_imp_reward_bounds():
    assert P.par_reward(7600, -2220) == 1.0 and P.par_reward(-7600, 2220) == -1.0
    assert P.par_reward(420, 300) == np.float32(3) / np.float32(24)


def _config(**kw):
    from brl_b200 import ppo
    cfg = ppo.default_config()
    cfg.update(kw)
    return cfg


@pytest.mark.parametrize("kw,match", [
    (dict(reward_mode="imp"), "reward_mode must be one of"),
    (dict(reward_mode="par_imp", game_mode="free-run"), "competitive"),
    (dict(reward_mode="par_imp", actor_illegal_action_mask=False, actor_illegal_action_penalty=True), "actor_illegal_action_mask"),
])
def test_bad_reward_modes_are_refused_before_any_device_work(kw, match):
    from brl_b200 import ppo
    from brl_b200.roll_out import check_reward_mode
    with pytest.raises(ValueError, match=match):
        check_reward_mode(_config(**kw))
    with pytest.raises(ValueError, match=match):  # Learner checks it first: no device is touched on this CPU machine
        ppo.train(kw, 0, device="cpu")
    with pytest.raises(ValueError, match=match):
        ppo.train_population([{}, kw], [0, 1], device="cpu")


def test_defaults_keep_the_score_reward():
    from brl_b200 import ppo
    from brl_b200.roll_out import check_reward_mode
    cfg = ppo.default_config()
    assert cfg["reward_mode"] == "score" and cfg["log_par"] is False
    check_reward_mode(cfg)
    check_reward_mode(_config(reward_mode="par_imp"))


def test_learners_may_pick_their_own_reward_mode_and_pbt_will_not_perturb_it():
    from brl_b200 import ppo
    from brl_b200.pbt import check_pbt_config
    from brl_b200.update import check_population_configs
    check_population_configs([ppo.full_config({}), ppo.full_config(dict(reward_mode="par_imp"))])
    with pytest.raises(ValueError, match="reward_mode"):
        check_pbt_config(dict(perturb_keys=("lr", "reward_mode")), 4)


def _bind(L, name):
    fn = getattr(L, name)
    fn.restype, fn.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]
    return fn


def test_par_ops_validate_their_arguments_without_a_gpu():
    from brl_b200 import _lib
    L = _lib.load()
    assert L.brl_xla_layout(b"brl_par") == b"iioo" and L.brl_xla_layout(b"brl_gather_reward_par") == b"iiiiox"
    for name in ("brl_par", "brl_gather_reward_par"):
        assert name in _lib.OPS and name in _lib.LAZY_OPS and name + "_xla" in _lib.XLA_LEGACY
    par, gather = _bind(L, "brl_par"), _bind(L, "brl_gather_reward_par")
    fake = lambda n, a=4096: (ctypes.c_void_p * n)(*[ctypes.c_void_p(a)] * n)  # noqa: E731 -- never dereferenced
    p = _lib.BrlParams(8, 0, 8, 0, 10, 0, 0, 0, -1.0, 1.0, 0.0, 0.0)
    assert par(None, fake(4), ctypes.byref(p), 8) == -1 and b"BrlParams" in L.brl_last_error()
    for k, name in enumerate((b"state", b"deal_table", b"par")):
        b = fake(4)
        b[k] = None
        assert par(None, b, ctypes.byref(p), ctypes.sizeof(p)) == -2
        assert b"brl_par: buffer '" + name + b"' is NULL" in L.brl_last_error()
    for k, name in ((0, b"state"), (2, b"par")):
        b = fake(4)
        b[k] = 4096 + 4
        assert par(None, b, ctypes.byref(p), ctypes.sizeof(p)) == -2
        assert b"brl_par: buffer '" + name + b"' is not 16-byte aligned" in L.brl_last_error()
    b = fake(4)
    b[3] = 4096 + 2
    assert par(None, b, ctypes.byref(p), ctypes.sizeof(p)) == -2 and b"'contract' is not 4-byte aligned" in L.brl_last_error()
    p.state_stride = 4
    assert par(None, fake(4), ctypes.byref(p), ctypes.sizeof(p)) == -1 and b"state_stride" in L.brl_last_error()
    names = (b"rewards", b"actor", b"par", b"done", b"reward")
    for k, name in enumerate(names):
        b = fake(6)
        b[k] = None
        assert gather(None, b, ctypes.byref(p), ctypes.sizeof(p)) == -2
        assert b"brl_gather_reward_par: buffer '" + name + b"' is NULL" in L.brl_last_error()
    for k, name in ((0, b"rewards"), (2, b"par")):
        b = fake(6)
        b[k] = 4096 + 4
        assert gather(None, b, ctypes.byref(p), ctypes.sizeof(p)) == -2
        assert b"buffer '" + name + b"' is not 16-byte aligned" in L.brl_last_error()
    p.flags = _lib.F_COUNT_DONE
    b = fake(6)
    b[5] = None
    assert gather(None, b, ctypes.byref(p), ctypes.sizeof(p)) == -2 and b"'count' is NULL" in L.brl_last_error()
    b[5] = 4096 + 4
    assert gather(None, b, ctypes.byref(p), ctypes.sizeof(p)) == -2 and b"'count' is not 8-byte aligned" in L.brl_last_error()
    stats = _bind(L, "brl_par_stats")
    assert L.brl_xla_layout(b"brl_par_stats") == b"iiiiiiiix" and "brl_par_stats" in _lib.LAZY_OPS
    p.flags = 0
    names = (b"state", b"deal_table", b"rewards_a", b"last_bid_a", b"last_bidder_a", b"rewards_b", b"last_bid_b",
             b"last_bidder_b", b"sums")
    for k, name in enumerate(names):
        b = fake(9)
        b[k] = None
        assert stats(None, b, ctypes.byref(p), ctypes.sizeof(p)) == -2
        assert b"brl_par_stats: buffer '" + name + b"' is NULL" in L.brl_last_error()
    for k in (0, 2, 5, 8):
        b = fake(9)
        b[k] = 4096 + 8
        assert stats(None, b, ctypes.byref(p), ctypes.sizeof(p)) == -2
        assert b"buffer '" + names[k] + b"' is not 16-byte aligned" in L.brl_last_error()
    p.n_envs = 0  # an empty batch is a no-op: NULL buffers are never looked at
    assert par(None, (ctypes.c_void_p * 4)(), ctypes.byref(p), ctypes.sizeof(p)) == 0
    assert gather(None, (ctypes.c_void_p * 6)(), ctypes.byref(p), ctypes.sizeof(p)) == 0
    assert stats(None, (ctypes.c_void_p * 9)(), ctypes.byref(p), ctypes.sizeof(p)) == 0
    p.n_envs = -1
    assert par(None, fake(4), ctypes.byref(p), ctypes.sizeof(p)) == -1 and b"n_envs" in L.brl_last_error()
