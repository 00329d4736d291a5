"""Golden vectors for BASELINE.json configs[0]: the `eval.py` duplicate match
`model-pretrained-rl.pkl` vs `model-sl.pkl`, num_eval_envs=100 (eval.py:28,43-65; src/evaluation.py:69-204).

Run where the reference tree is available (its path is the first argument):

    python tests/golden/make_c1_golden.py /path/to/reference            # -> c1_eval_match.npz
    python tests/golden/make_c1_golden.py /path/to/reference --seeded   # -> c1_seeded_match.npz

What it does
  * loads the two BUNDLED pickles (bridge_models/, real trained weights) without jax;
  * plays the 100-env match on the CPU oracle (oracle/brl_oracle.c) over the 1000 real boards + double-dummy tables of
    wb5/dataset_for_vs_wb5.json (the pgx DDS file `dds_results/test_000.npy` eval.py:43 opens is a download and absent),
    every decision = masked argmax of a FLOAT64 NumPy evaluation of the DeepMind MLP (src/models.py:23-33,
    src/evaluation.py:124-151: team 1 = players 0/1, team 2 = players 2/3);
  * cross-checks every board's IMPs with the reference's OWN code: the two auctions go through the JSON board-log
    format into `JsonParser`, `calc_score` and `score_to_imp` (wb5/analyze_log.py:63-155);
  * freezes per-step actions, liveness, float64 top-2 logit gaps (how close each decision is to a tie), per-board IMPs,
    both tables' final contracts and mean / SE / win-rate into tests/golden/c1_eval_match.npz;
  * copies the five bundled weight files to tests/golden/_weights/ (git-ignored: 15 MB each).
With --seeded the same match is played by the two seeded nets of tests/helpers.seeded_params (SEEDED_WEIGHTS) instead of
the bundled pickles, so that the repository alone can check a whole match against the reference's scorer.
"""
import os
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
WEIGHTS = os.path.join(HERE, "_weights")
MODELS = ("model-pretrained-rl.pkl", "model-sl.pkl", "model-from-scratch-rl.pkl", "model-pretrained-rl-with-fsp.pkl",
          "model-pretrained-rl-with-pfsp.pkl")
SEEDED_WEIGHTS = (1, 2)


def copy_weights(ref):
    os.makedirs(WEIGHTS, exist_ok=True)
    for name in MODELS:
        dst = os.path.join(WEIGHTS, name)
        src = os.path.join(ref, "bridge_models", name)
        if not os.path.exists(dst) or os.path.getsize(dst) != os.path.getsize(src):
            shutil.copyfile(src, dst)


def mlp64(p, x):
    h = np.asarray(x, np.float64)
    for i in range(4):
        h = np.maximum(h @ p[f"w{i}"].astype(np.float64) + p[f"b{i}"].astype(np.float64), 0.0)
    return h @ p["w4"].astype(np.float64) + p["b4"].astype(np.float64)


def main(ref, seeded):
    from brl_b200 import board_log
    from brl_b200 import random as brandom
    from brl_b200.models import load_params, params_to_numpy
    from oracle import oracle as orc
    from tests import helpers as H
    if seeded:
        p1, p2 = (params_to_numpy(H.seeded_params(s, "cpu")) for s in SEEDED_WEIGHTS)
    else:
        copy_weights(ref)
        p1 = params_to_numpy(load_params(os.path.join(WEIGHTS, MODELS[0]), "cpu"))
        p2 = params_to_numpy(load_params(os.path.join(WEIGHTS, MODELS[1]), "cpu"))
    boards = H.load_boards()
    n = 100
    rng = brandom.PRNGKey(0)                      # eval.py:44
    _, sub = brandom.split(rng)                   # src/evaluation.py:93
    env = orc.OracleEnv(boards["table"], n)
    env.init(orc.make_keys(sub, n))
    priv0 = env.export_private()
    env.duplicate_tables_from_state()
    cum = np.zeros(n, np.float64)
    actions, lives, gaps, record = [], [], [], []
    for step in range(400):
        e = env.export()
        if e["terminated"].all():
            break
        live = e["terminated"] == 0
        lg = np.where((e["current_player"] < 2)[:, None], mlp64(p1, e["observation"]), mlp64(p2, e["observation"]))
        masked = np.where(e["legal_action_mask"] != 0, lg, -np.inf)
        act = masked.argmax(1).astype(np.int32)   # first argmax = distrax mode (src/evaluation.py:131-133)
        top2 = np.sort(masked, axis=1)[:, -2:]
        gap = np.where(np.isfinite(top2[:, 0]), top2[:, 1] - top2[:, 0], np.inf)
        record.append((act.copy(), env.info_a["terminated"].copy(), env.info_b["terminated"].copy()))
        actions.append(act); lives.append(live.astype(np.uint8)); gaps.append(np.where(live, gap, np.inf))
        env.duplicate_step(act)
        cum += env.export()["rewards"][:, 0]
    assert env.export()["terminated"].all()
    mean, se, win = orc.match_stats(cum)

    # ---- the reference's own parser / scorer must reproduce every board's IMPs ------------------------------------
    t1, t2 = board_log.match_to_board_logs(boards["table"], priv0["deal"], priv0["dealer"], priv0["vul"],
                                           priv0["shuffled_players"], record, team_names=("team1", "team2"),
                                           board_ids=[str(i) for i in range(n)])
    import tempfile
    sys.path.insert(0, os.path.join(ref, "submodule", "bridge_env"))
    from bridge_env import Pair, Player
    from bridge_env.data_handler.json_handler.parser import JsonParser
    from bridge_env.score import calc_score, score_to_imp
    with tempfile.TemporaryDirectory() as tmp:
        parsed = []
        for name, entries in (("t1.json", t1), ("t2.json", t2)):
            with open(os.path.join(tmp, name), "w") as fh:
                board_log.write_logs(fh, entries)
            with open(os.path.join(tmp, name)) as fh:
                parsed.append(JsonParser().parse_board_logs(fh))

    def team1_score(d):                           # wb5/analyze_log.py:86-95,131-147, oriented to team 1
        if d.contract.is_passed_out():
            return 0
        s = calc_score(d.contract, d.dda[d.declarer][d.contract.trump])
        pair = Pair.NS if d.players[Player.N] == "team1" else Pair.EW
        return s if d.declarer.pair is pair else -s

    for i, (d1, d2) in enumerate(zip(*parsed)):
        assert score_to_imp(team1_score(d1), team1_score(d2)) == int(cum[i]), f"board {i}: reference scorer disagrees"

    g = np.stack(gaps)
    out = dict(
        n=np.int32(n), seed=np.int64(0), actions=np.stack(actions).astype(np.int8), live=np.stack(lives),
        gap=g.astype(np.float32), imps=cum.astype(np.float32), stats=np.array([mean, se, win], np.float64),
        a_last_bid=env.info_a["last_bid"].astype(np.int32), a_last_bidder=env.info_a["last_bidder"].astype(np.int32),
        a_rewards=env.info_a["rewards"].astype(np.float32), b_last_bid=env.info_b["last_bid"].astype(np.int32),
        b_last_bidder=env.info_b["last_bidder"].astype(np.int32), b_rewards=env.info_b["rewards"].astype(np.float32),
        deal=priv0["deal"].astype(np.int32), dealer=priv0["dealer"].astype(np.int32))
    if seeded:
        out["weight_seeds"] = np.array(SEEDED_WEIGHTS, np.int64)
    else:
        out["models"] = np.array(MODELS[:2])
    np.savez_compressed(os.path.join(HERE, "c1_seeded_match.npz" if seeded else "c1_eval_match.npz"), **out)
    fin = g[np.isfinite(g)]
    print(f"C1 golden: {len(actions)} steps, {int(np.stack(lives).sum())} live decisions, IMP {mean:.4f} +- {se:.4f}, "
          f"win rate {win:.3f}; smallest top-2 gap {fin.min():.3e}, decisions with gap <= 1e-4: {(fin <= 1e-4).sum()}")


if __name__ == "__main__":
    main(sys.argv[1], "--seeded" in sys.argv[2:])
