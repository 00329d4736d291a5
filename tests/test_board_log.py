"""CPU: board logs of a duplicate match (brl_b200/board_log.py) in the reference's JSON format.
A match is played on the oracle env with random-legal actions; the written files are then read
back (a) structurally, against the golden score table, and (b) against what the reference's OWN
`JsonParser`, `calc_score` and `score_to_imp` (wb5/analyze_log.py:63-155) read from the same
logs, frozen in tests/golden/board_log_ref.npz, whose IMPs must equal the env's."""
import io
import json
import os

import numpy as np
import pytest

from brl_b200 import board_log
from brl_b200 import deals
from oracle import oracle as orc
from tests import helpers as H


def _play_match(n=200, seed=5):
    boards = H.load_boards()
    env = orc.OracleEnv(boards["table"], n)
    env.init(orc.make_keys(seed, n))
    priv0 = env.export_private()
    env.duplicate_tables_from_state()
    record, cum = [], np.zeros(n)
    for step in range(400):
        a_term, b_term = env.info_a["terminated"].copy(), env.info_b["terminated"].copy()
        if env.export()["terminated"].all():
            break
        action = env.random_legal_actions(seed, step)
        record.append((action, a_term, b_term))
        env.duplicate_step(action)
        cum += env.export()["rewards"][:, 0]
    assert env.export()["terminated"].all()
    return boards, env, priv0, record, cum


def test_score_closed_form_matches_golden_table():
    tab = np.load(H.GOLDEN + "/score_table.npy")
    for b in range(35):
        for d, (x, xx) in enumerate(((0, 0), (1, 0), (1, 1))):
            for v in (0, 1):
                for t in range(14):
                    assert board_log.contract_score(b, bool(x), bool(xx), bool(v), t) == tab[b, d, v, t]


def test_known_auction_contract_and_strings():
    known = H.load_known()
    # wb5/utils.py:60-68 auction + 'Pass': 6C by E (tests/test_bidding_phase.py:28-68 shape)
    calls = [0, 9, 11, 20, 1, 0, 22, 1, 2, 0, 0, 28, 0, 0, 0]
    last_bid, x, xx, declarer = board_log.resolve_contract(calls, dealer=2)
    assert (last_bid, x, xx) == (25, False, False) and board_log.ACTION_STR[28] == "6C"
    assert board_log.SEATS[declarer] == "E"                      # SURVEY B.2: 6C by E
    assert board_log.resolve_contract([0, 0, 0, 0], 1) == (None, False, False, None)
    assert [board_log.ACTION_STR[a] for a in (0, 1, 2, 3, 7, 37)] == ["Pass", "X", "XX", "1C", "1NT", "7NT"]
    assert known is not None


def test_match_logs_roundtrip_and_scores():
    boards, env, priv0, record, cum = _play_match()
    t1, t2 = board_log.match_to_board_logs(boards["table"], priv0["deal"], priv0["dealer"], priv0["vul"],
                                           priv0["shuffled_players"], record, team_names=("actor", "opp"))
    buf = io.StringIO()
    board_log.write_logs(buf, t1)
    back = json.loads(buf.getvalue())["logs"]
    assert back == t1 and len(t1) == len(t2) == 200
    owners, dd = deals.unpack_deal_table(boards["table"])
    for i, (e1, e2) in enumerate(zip(t1, t2)):
        # same board at both tables, seats swapped between the teams
        assert e1["deal"] == e2["deal"] and e1["dealer"] == e2["dealer"] and e1["vulnerability"] == e2["vulnerability"]
        assert all(e1["players"][s] != e2["players"][s] for s in "NESW")
        assert e1["players"]["N"] == e1["players"]["S"] != e1["players"]["E"] == e1["players"]["W"]
        assert sorted(sum(e1["deal"].values(), [])) == sorted(board_log._card_str(c) for c in range(52))
        # the env's own terminal info agrees with the log text
        for e, info in ((e1, env.info_a[i]), (e2, env.info_b[i])):
            if e["contract"] == "Passed_out":
                assert info["last_bid"] == -1 and e["declarer"] is None and e["taken_trick"] is None
            else:
                assert e["contract"].rstrip("X") == board_log.ACTION_STR[info["last_bid"] + 3]
                assert e["contract"].endswith("XX") == bool(info["call_xx"])
                ns_team = 0 if e["players"]["N"] == "actor" else 1
                want_ns = info["rewards"][0] if ns_team == 0 else info["rewards"][2]
                assert e["scores"]["NS"] == int(want_ns)
        # IMPs of team "actor" from the two logs == the env's duplicate reward (src/duplicate.py:46-70)
        s1 = e1["scores"]["NS"] if e1["players"]["N"] == "actor" else e1["scores"]["EW"]
        s2 = e2["scores"]["NS"] if e2["players"]["N"] == "actor" else e2["scores"]["EW"]
        assert orc.imp(s1 + s2) == int(cum[i])


def test_reference_parser_and_analysis_accept_the_logs():
    """The logs of this match, as the reference's `JsonParser`, `calc_score` and `score_to_imp` read them
    (wb5/analyze_log.py:63-155, scores oriented to team "actor"), are frozen in tests/golden/board_log_ref.npz by
    tests/golden/make_board_log_golden.py.  The logs written now must say the same and give the env's IMPs."""
    boards, env, priv0, record, cum = _play_match(n=120, seed=8)
    logs = board_log.match_to_board_logs(boards["table"], priv0["deal"], priv0["dealer"], priv0["vul"],
                                         priv0["shuffled_players"], record, team_names=("actor", "opp"),
                                         board_ids=[str(i) for i in range(120)])
    ref = np.load(os.path.join(H.GOLDEN, "board_log_ref.npz"))
    written = []
    for entries in logs:
        buf = io.StringIO()
        board_log.write_logs(buf, entries)
        written.append(json.loads(buf.getvalue())["logs"])
    for i in range(120):
        assert int(ref["imp"][i]) == int(cum[i]), f"board {i}"
        for t in range(2):
            e = written[t][i]
            assert " ".join(e["bid_history"]) == ref["bid_history"][t, i], f"board {i} table {t + 1}"
            assert (e["declarer"] or "") == ref["declarer"][t, i], f"board {i} table {t + 1}"
            if e["declarer"] is not None:
                assert e["contract"] == ref["contract"][t, i], f"board {i} table {t + 1}"
            actor_side = "NS" if e["players"]["N"] == "actor" else "EW"
            assert e["scores"][actor_side] == int(ref["score"][t, i]), f"board {i} table {t + 1}"


@pytest.mark.gpu
def test_gpu_match_record_to_board_logs_and_reference_parser():
    """SURVEY 8f-4 on the GPU path: a duplicate match played by the CUDA kernels (`record=` of
    make_simple_duplicate_evaluate: per step the action and both tables' terminated flags), written as the reference's
    JSON board logs.  The logs' own scores must give the GPU match's IMPs board by board, and so must the reference's
    `calc_score` + `score_to_imp` (wb5/analyze_log.py:131-147) applied to the written logs."""
    import torch
    from brl_b200 import BridgeBidding
    from brl_b200 import random as brandom
    from brl_b200.evaluation import make_simple_duplicate_evaluate
    from brl_b200.models import init_params
    dev = "cuda:0"
    boards = H.load_boards()
    env = BridgeBidding(table=boards["table"], device=dev)
    n = 150
    rng = brandom.PRNGKey(21)
    _, sub = brandom.split(rng)
    state0 = env.init(env.make_keys(sub, n))          # the same draws the evaluator makes: private fields of the start state
    priv = {k: getattr(state0, "_" + k).cpu().numpy() for k in ("deal", "dealer", "shuffled_players")}
    vul = np.stack([state0._vul_NS.cpu().numpy(), state0._vul_EW.cpu().numpy()], axis=1).astype(np.uint8)
    evaluate = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)
    record = []
    (mean, se, win), info_a, info_b, cum = evaluate(init_params(5, dev), init_params(6, dev), rng, record=record)
    cum = cum.cpu().numpy()
    t1, t2 = board_log.match_to_board_logs(boards["table"], priv["deal"], priv["dealer"], vul, priv["shuffled_players"], record,
                                           team_names=("actor", "opp"), board_ids=[str(i) for i in range(n)])
    assert len(t1) == len(t2) == n
    for i, (e1, e2) in enumerate(zip(t1, t2)):
        s1 = e1["scores"]["NS"] if e1["players"]["N"] == "actor" else e1["scores"]["EW"]
        s2 = e2["scores"]["NS"] if e2["players"]["N"] == "actor" else e2["scores"]["EW"]
        assert orc.imp(s1 + s2) == int(cum[i]), f"board {i}"
        for e, info_bid in ((e1, int(info_a.last_bid[i])), (e2, int(info_b.last_bid[i]))):
            if e["contract"] == "Passed_out":
                assert info_bid == -1
            else:
                assert e["contract"].rstrip("X") == board_log.ACTION_STR[info_bid + 3]
    assert abs(mean - float(cum.astype(np.float64).mean())) < 1e-9
    # the reference's scorer as frozen in the golden tables (calc_bid_score -> score_table.npy, score_to_imp(d, 0) ->
    # imp_table.npy, tests/golden/make_golden.py): each written log's contract, vulnerability and double-dummy tricks
    # scored as wb5/analyze_log.py:131-147 does, oriented to team "actor", must give the GPU match's IMPs board by board
    score_tab, imp_tab = np.load(H.GOLDEN + "/score_table.npy"), np.load(H.GOLDEN + "/imp_table.npy")

    def actor_score(e):
        if e["contract"] == "Passed_out":
            return 0
        bid = board_log.ACTION_STR.index(e["contract"].rstrip("X")) - 3
        doubled = len(e["contract"]) - len(e["contract"].rstrip("X"))
        pair = "NS" if e["declarer"] in "NS" else "EW"
        tricks = e["dda"][e["declarer"]][board_log.STRAINS[bid % 5]]
        s = int(score_tab[bid, doubled, int(e["vulnerability"] in (pair, "Both")), tricks])
        return s if e["players"][pair[0]] == "actor" else -s

    written = []
    for entries in (t1, t2):
        buf = io.StringIO()
        board_log.write_logs(buf, entries)
        written.append(json.loads(buf.getvalue())["logs"])
    assert (imp_tab[:401] == -24).all() and (imp_tab[1200:] == 24).all()    # 24 IMPs from 4000 points on
    for i, (e1, e2) in enumerate(zip(*written)):
        d = min(max(actor_score(e1) + actor_score(e2), -8000), 8000)
        assert int(imp_tab[(d + 8000) // 10]) == int(cum[i]), f"board {i}"
