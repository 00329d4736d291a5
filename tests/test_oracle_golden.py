"""CPU: pin the oracle (oracle/brl_oracle.c) against golden vectors produced by the
reference's own Python (tests/golden/make_golden.py).  No GPU needed."""
import numpy as np
import pytest

from oracle import oracle as orc
from tests import helpers as H


def test_score_table_matches_reference_calc_bid_score():
    # submodule/bridge_env/tests/test_score.py:130-163 enumerates the same grid
    tab = np.load(H.GOLDEN + "/score_table.npy")
    for b in range(35):
        for d, (x, xx) in enumerate(((0, 0), (1, 0), (1, 1))):
            for v in (0, 1):
                for t in range(14):
                    assert orc.score(b, x, xx, v, t) == tab[b, d, v, t], (b, d, v, t)
    assert tab.min() == -7600 and abs(tab).max() == 7600  # reward_scale = 7600 (ppo.py:174)


def test_imp_table_matches_reference_score_to_imp():
    tab = np.load(H.GOLDEN + "/imp_table.npy")
    got = np.array([orc.imp(d) for d in range(-8000, 8001, 10)])
    assert (got == tab).all()


@pytest.mark.parametrize("a,b,want", [
    ([0, 0, 0, 0], [0, 0, 0, 0], [0, 0, 0, 0]),
    ([0, 0, 0, 0], [100, 100, -100, -100], [3, 3, -3, -3]),
    ([-100, -100, 100, 100], [0, 0, 0, 0], [-3, -3, 3, 3]),
    ([-100, -100, 100, 100], [100, 100, -100, -100], [0, 0, 0, 0]),
    ([-3500, -3500, 3500, 3500], [0, 0, 0, 0], [-23, -23, 23, 23]),
    ([2000, 2000, -2000, -2000], [2000, 2000, -2000, -2000], [24, 24, -24, -24]),
])
def test_imp_reward_doctests(a, b, want):
    # src/duplicate.py:20-43
    assert orc.imp_reward(a, b).tolist() == [float(w) for w in want]


def _run_golden_auctions(seating_of_auction):
    boards = H.load_boards()
    gold = H.load_auctions()
    calls, lens = H.auction_matrix(gold)
    n = len(lens)
    players = H.SEATINGS[seating_of_auction(n)]
    env = orc.OracleEnv(boards["table"], n)
    env.reset_fields(gold["board"], gold["dealer"], gold["vul_ns"], gold["vul_ew"], players)
    want_obs = H.unpack_obs_bits(gold["obs_bits"])
    off = gold["offsets"]
    total_r = np.zeros((n, 4), np.float32)
    for k in range(calls.shape[1]):
        live = np.flatnonzero(lens > k)
        out = env.export(np.uint8)
        rows = off[live] + k
        assert (out["observation"][live] == want_obs[rows]).all(), f"obs mismatch at call {k}"
        assert (out["legal_action_mask"][live] == gold["mask"][rows]).all(), f"mask mismatch at call {k}"
        assert (out["terminated"][live] == 0).all()
        # the player to act sits at seat (dealer + k) % 4
        seat = (gold["dealer"][live].astype(int) + k) % 4
        assert (out["current_player"][live] == players[live, seat]).all()
        env.step(np.where(lens > k, calls[:, k], 0).astype(np.int32))
        step_out = env.export(np.uint8)
        # rewards are non-zero only on the terminal step; finished envs no-op with zeros
        assert (step_out["rewards"][lens != k + 1] == 0).all()
        assert (step_out["terminated"] == (lens <= k + 1)).all()
        total_r += step_out["rewards"]
    out = env.export(np.uint8)
    assert (out["terminated"] == 1).all()
    want_r = np.stack([H.expected_rewards(gold["final"][i], players[i]) for i in range(n)])
    assert (total_r == want_r).all()
    priv = env.export_private()
    bid = gold["final"][:, 1]
    assert (priv["last_bid"] == bid).all()
    has = bid >= 0
    assert (priv["call_x"][has] == gold["final"][has, 2]).all()
    assert (priv["call_xx"][has] == gold["final"][has, 3]).all()
    assert (priv["step_count"] == lens).all()
    # stepping a finished env is a zero-reward no-op (src/evaluation.py:120-122)
    env.step(np.zeros(n, np.int32))
    out2 = env.export(np.uint8)
    assert (out2["rewards"] == 0).all() and (out2["terminated"] == 1).all()
    assert (out2["observation"] == out["observation"]).all()


def test_oracle_matches_reference_on_2000_auctions_fixed_seating():
    _run_golden_auctions(lambda n: np.zeros(n, dtype=int))


def test_oracle_matches_reference_on_2000_auctions_all_seatings():
    _run_golden_auctions(lambda n: np.arange(n) % 8)


def test_known_auction_bits_from_wb5_utils_selfcheck():
    # wb5/utils.py:54-89: dealer E, vul None; history bit indices = SURVEY Appendix B.1
    known = H.load_known()["wb5_utils_14call_plus_final_pass"]
    boards = H.load_boards()
    env = orc.OracleEnv(boards["table"], 1)
    env.reset_fields([known["board"]], [known["dealer"]], [0], [0], H.SEATINGS[[4]])  # [0,3,1,2] wb5/utils.py:72
    for k, a in enumerate(known["calls"]):
        out = env.export(np.uint8)
        assert np.flatnonzero(out["observation"][0]).tolist() == known["set_bits"][k]
        assert int(out["legal_action_mask"][0].sum()) == known["n_legal"][k]
        env.step(np.array([a], np.int32))
    out = env.export()
    assert out["terminated"][0] == 1
    # 6C by N (seat 0 = player 0), DD tricks 11 -> one down, not vulnerable: -50 for team {0,1}
    assert out["rewards"][0].tolist() == [-50.0, -50.0, 50.0, 50.0]


def test_known_auction_test_bidding_phase1_illegal_probes():
    # submodule/bridge_env/tests/test_bidding_phase.py:28-68
    known = H.load_known()["test_bidding_phase1"]
    boards = H.load_boards()
    env = orc.OracleEnv(boards["table"], 1)
    env.reset_fields([0], [known["dealer"]], [known["vul_ns"]], [known["vul_ew"]], H.SEATINGS[[0]])
    for a in known["calls"][:-1]:
        env.step(np.array([a], np.int32))
    mask = env.export()["legal_action_mask"][0]
    for a in known["illegal_before_final_pass"]:
        assert mask[a] == 0
    env.step(np.array([known["calls"][-1]], np.int32))
    assert env.export()["terminated"][0] == 1
    decl, bid, x, xx, vul, _ = known["final"]
    assert (decl, bid // 5 + 1, bid % 5, vul) == (1, 6, 0, 0)  # E declares 6C, not vulnerable


def test_pass_out_gives_zero_rewards():
    # submodule/bridge_env/tests/test_bidding_phase.py:7-26; src/evaluation.py:465-467
    boards = H.load_boards()
    env = orc.OracleEnv(boards["table"], 1)
    env.reset_fields([3], [2], [1], [1], H.SEATINGS[[1]])
    for _ in range(3):
        env.step(np.zeros(1, np.int32))
        assert env.export()["terminated"][0] == 0
    env.step(np.zeros(1, np.int32))
    out, priv = env.export(), env.export_private()
    assert out["terminated"][0] == 1 and (out["rewards"] == 0).all()
    assert priv["last_bid"][0] == -1 and priv["last_bidder"][0] == -1 and priv["pass_num"][0] == 4


def test_illegal_action_terminates_with_penalty():
    boards = H.load_boards()
    env = orc.OracleEnv(boards["table"], 1)
    env.reset_fields([3], [0], [0], [0], H.SEATINGS[[0]])
    env.step(np.array([1], np.int32))  # X before any bid
    out = env.export()
    assert out["terminated"][0] == 1
    assert out["rewards"][0].tolist() == [-1.0, 1.0, 1.0, 1.0]


def test_c1_golden_match_replays_on_the_oracle():
    """configs[0] (eval.py: model-pretrained-rl vs model-sl, 100 envs): the frozen action sequence (made with a float64
    MLP and checked board by board against the reference's own JsonParser / calc_score / score_to_imp by
    tests/golden/make_c1_golden.py) replayed through the C oracle gives the frozen IMPs, contracts and statistics; and,
    where the bundled weights have been copied in, the oracle's fp32 NumPy MLP on them takes the same decisions."""
    from brl_b200.models import load_params, params_to_numpy
    g = H.load_c1()
    try:
        nets = [params_to_numpy(load_params(H.weight_path(str(m)), "cpu")) for m in g["models"]]
    except FileNotFoundError:
        nets = None  # the bundled weights are not in the repository: the env-side replay below still runs
    _replay_c1_on_the_oracle(g, nets)


def test_c1_seeded_match_replays_on_the_oracle():
    """The same match played by the two seeded nets of tests/helpers.seeded_params (tests/golden/make_c1_golden.py
    --seeded, checked against the reference's own scorer): replayed through the C oracle it gives the frozen IMPs,
    contracts and statistics, and the oracle's fp32 NumPy MLP on the seeded nets takes the same decisions."""
    from brl_b200.models import params_to_numpy
    g = H.load_c1_seeded()
    _replay_c1_on_the_oracle(g, [params_to_numpy(H.seeded_params(int(s), "cpu")) for s in g["weight_seeds"]])


def _replay_c1_on_the_oracle(g, nets):
    from brl_b200 import random as brandom
    from oracle import oracle as orc
    boards = H.load_boards()
    n = int(g["n"])
    _, sub = brandom.split(brandom.PRNGKey(int(g["seed"])))
    env = orc.OracleEnv(boards["table"], n)
    env.init(orc.make_keys(sub, n))
    priv = env.export_private()
    assert (priv["deal"] == g["deal"]).all() and (priv["dealer"] == g["dealer"]).all()
    env.duplicate_tables_from_state()
    cum = np.zeros(n)
    for t in range(g["actions"].shape[0]):
        e = env.export()
        live = e["terminated"] == 0
        assert (live.astype(np.uint8) == g["live"][t]).all()
        if nets is not None:
            lg = np.where((e["current_player"] < 2)[:, None], orc.mlp_forward(nets[0], e["observation"])[0],
                          orc.mlp_forward(nets[1], e["observation"])[0])
            act, _ = orc.categorical(lg, e["legal_action_mask"], sample=False)
            assert (act[live] == g["actions"][t][live]).all()      # smallest float64 top-2 gap: 1.4e-3 (bundled), 3.7e-3 (seeded)
        env.duplicate_step(g["actions"][t].astype(np.int32))
        cum += env.export()["rewards"][:, 0]
    assert env.export()["terminated"].all()
    assert (cum == g["imps"]).all()
    np.testing.assert_allclose(orc.match_stats(cum), g["stats"], rtol=1e-12)
    for k, info in (("a", env.info_a), ("b", env.info_b)):
        assert (info["last_bid"] == g[k + "_last_bid"]).all() and (info["last_bidder"] == g[k + "_last_bidder"]).all()
        assert (info["rewards"] == g[k + "_rewards"]).all()
    assert float(g["gap"][np.isfinite(g["gap"])].min()) > 1e-4
