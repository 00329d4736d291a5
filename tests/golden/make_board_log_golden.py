"""Golden vectors for tests/test_board_log.py: the reference's own reading of the board logs of one seeded match.

Run where the reference tree is available (its path is the first argument):

    python tests/golden/make_board_log_golden.py /path/to/reference

The match of `test_reference_parser_and_analysis_accept_the_logs` (120 boards, oracle env, random-legal actions, seed 8)
is written as JSON board logs and read back by the reference's `JsonParser`; each board is scored with its `calc_score`
and `score_to_imp` following wb5/analyze_log.py:63-155, oriented to team "actor".  What the parser and scorer returned
is frozen into board_log_ref.npz, so that the test keeps comparing the logs with the reference without it:
  contract, declarer, bid_history   str[2, 120]   table 1 / table 2 as the parser read them ("" = no declarer)
  score                             int32[2, 120] calc_score of the contract at the double-dummy tricks, actor's sign
  imp                               int32[120]    score_to_imp(table 1, table 2)
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

N_BOARDS, SEED = 120, 8


def main(ref):
    from brl_b200 import board_log
    from tests.test_board_log import _play_match
    boards, env, priv0, record, cum = _play_match(n=N_BOARDS, seed=SEED)
    logs = board_log.match_to_board_logs(boards["table"], priv0["deal"], priv0["dealer"], priv0["vul"],
                                         priv0["shuffled_players"], record, team_names=("actor", "opp"),
                                         board_ids=[str(i) for i in range(N_BOARDS)])
    sys.path.insert(0, os.path.join(ref, "submodule", "bridge_env"))
    from bridge_env import Pair, Player
    from bridge_env.data_handler.json_handler.parser import JsonParser
    from bridge_env.score import calc_score, score_to_imp
    parsed = []
    with tempfile.TemporaryDirectory() as tmp:
        for name, entries in zip(("t1.json", "t2.json"), logs):
            with open(os.path.join(tmp, name), "w") as fh:
                board_log.write_logs(fh, entries)
            with open(os.path.join(tmp, name)) as fh:
                parsed.append(JsonParser().parse_board_logs(fh))

    def actor_score(d):                                # wb5/analyze_log.py:86-95,131-147, oriented to team "actor"
        if d.contract.is_passed_out():
            return 0
        s = calc_score(d.contract, d.dda[d.declarer][d.contract.trump])
        return s if d.declarer.pair is (Pair.NS if d.players[Player.N] == "actor" else Pair.EW) else -s

    out = dict(contract=np.array([[str(d.contract) for d in t] for t in parsed]),
               declarer=np.array([["" if d.declarer is None else str(d.declarer) for d in t] for t in parsed]),
               bid_history=np.array([[" ".join(str(b) for b in d.bid_history) for d in t] for t in parsed]),
               score=np.array([[actor_score(d) for d in t] for t in parsed], np.int32))
    out["imp"] = np.array([score_to_imp(int(a), int(b)) for a, b in zip(*out["score"])], np.int32)
    assert (out["imp"] == cum).all(), "the reference's IMPs differ from the env's"
    np.savez_compressed(os.path.join(HERE, "board_log_ref.npz"), **out)
    print(f"board-log golden: {N_BOARDS} boards, IMP sum {int(out['imp'].sum())}")


if __name__ == "__main__":
    main(sys.argv[1])
