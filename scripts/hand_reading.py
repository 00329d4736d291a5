"""Hand reading (DESIGN.md f18): how much each net's auctions tell its partner (and the opponents) about the hidden hands.

    python scripts/hand_reading.py [nets=a.pkl,b.pkl | seeds=1,2] [deals=dds_results/test_000.npy] boards=1000 \
        [samples=1024] [temperature=1] [at=end|decisions] [precision=tc|tc-bf16] [method=is|smc] [moves=1] \
        [ess_threshold=0.5] [out=hand_reading.json]
    python scripts/hand_reading.py data=test.txt nets=a.pkl [max_auctions=1000] ...
    python scripts/hand_reading.py hand=AKQ2.AK32.K32.32 auction=1C,P,1H dealer=N vul=NS observer=S nets=a.pkl

Sources: a duplicate match of net 0 against net 1 (nets= .pkl files, or seeded nets of the bundled architecture from seeds=)
on `boards` boards of the deal table `deals=` (synthetic when omitted), both tables played by the host match loop with
`record=`; or the auctions of an OpenSpiel data file (data=; dealer North, nobody vulnerable), every seat played by net 0.
Every auction is read by each of its four seats (at=end: after the last call; at=decisions: before each of the seat's own
calls) and scored per observer net (posterior.reading_stats).  method=smc reads them with the resample-move SMC sampler
(DESIGN.md f19: `moves` Metropolis-Hastings moves after each resample, resampling below ess_threshold x samples).  Writes the
JSON report.

With hand= (PBN order spades.hearts.diamonds.clubs, e.g. AKQ2.AK32.K32.32), auction= (comma-separated: P, X, XX, 1C .. 7NT),
dealer=, vul= (None, NS, EW, Both) and observer= it prints posterior.describe for that one hand instead, every seat played by
net 0; the other 39 cards of the one-row deal table are placeholders (they are what is sampled).
"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

DEFAULTS = dict(nets="", seeds="1,2", deals="", boards=1000, data="", max_auctions=1000, samples=1024, seed=0, temperature=1.0,
                at="end", precision="tc", row_budget=1 << 20, out="hand_reading.json", hand="", auction="", dealer="N",
                vul="None", observer="S", method="is", moves=1, ess_threshold=0.5)
CALLS = ["P", "X", "XX"] + [f"{lvl}{s}" for lvl in range(1, 8) for s in ("C", "D", "H", "S", "NT")]
RANKS = "23456789TJQKA"


def parse_args(argv):
    cfg = dict(DEFAULTS)
    for arg in argv:
        key, sep, value = arg.partition("=")
        if not sep or key not in cfg:
            raise SystemExit(f"expected key=value with key in {sorted(cfg)}, got {arg!r}")
        cfg[key] = type(DEFAULTS[key])(value)
    if bool(cfg["hand"]) != bool(cfg["auction"]):
        raise SystemExit("hand= and auction= go together")
    if cfg["at"] not in ("end", "decisions") or cfg["precision"] not in ("tc", "tc-bf16"):
        raise SystemExit("at= must be end or decisions, precision= tc or tc-bf16")
    if cfg["method"] not in ("is", "smc") or not 0 <= cfg["moves"] <= 64 or not 0.0 <= cfg["ess_threshold"] <= 1.0:
        raise SystemExit("method= must be is or smc, moves= in [0, 64], ess_threshold= in [0, 1]")
    return cfg


def one_hand_query(cfg):
    """(one-row deal table, calls, dealer, vul bits, observer seat) of the hand= / auction= / dealer= / vul= / observer= query"""
    from brl_b200.deals import pack_deal_table
    s = "NESW".index(cfg["observer"])
    suits = cfg["hand"].upper().split(".")
    if len(suits) != 4:
        raise SystemExit("hand= is four suits, spades.hearts.diamonds.clubs")
    own = [RANKS.index(r) * 4 + (3 - k) for k, suit in enumerate(suits) for r in suit]
    if len(own) != 13 or len(set(own)) != 13:
        raise SystemExit("hand= must hold 13 different cards")
    others = [c for c in range(52) if c not in own]
    owners = np.zeros(52, np.int64)
    owners[own] = s
    for k, c in enumerate(others):
        owners[c] = (s + 1 + k // 13) % 4
    calls = [CALLS.index(x.strip().upper()) for x in cfg["auction"].split(",") if x.strip()]
    vul = {"NONE": 0, "NS": 1, "EW": 2, "BOTH": 3}[cfg["vul"].upper()]
    return pack_deal_table(owners[None], np.zeros((1, 4, 5), np.int64)), calls, "NESW".index(cfg["dealer"]), vul, s


def load_nets(cfg, device):
    from brl_b200.models import load_params
    from tests.helpers import seeded_params
    if cfg["nets"]:
        return [load_params(p, device) for p in cfg["nets"].split(",") if p]
    return [seeded_params(int(x), device) for x in cfg["seeds"].split(",")]


def main(argv):
    cfg = parse_args(argv)
    from brl_b200 import posterior
    from brl_b200.deals import load_table, synthetic_deal_table
    dev = "cuda"
    nets = load_nets(cfg, dev)
    kw = dict(samples=cfg["samples"], seed=cfg["seed"], temperature=cfg["temperature"], row_budget=cfg["row_budget"],
              precision=None if cfg["precision"] == "tc" else cfg["precision"], method=cfg["method"], moves=cfg["moves"],
              ess_threshold=cfg["ess_threshold"])
    if cfg["hand"]:
        table, calls, dealer, vul, s = one_hand_query(cfg)
        post = posterior.hand_posterior(nets[:1], table, np.array(calls, np.uint8), [0, len(calls)], [[0, s, len(calls)]],
                                        [[0, 0, 0, 0]], dealer=[dealer], vul=[vul], **kw)
        print("\n".join(posterior.describe(post, 0)))
        return
    if cfg["data"]:
        from brl_b200 import sl
        traj = sl.parse_trajectories(cfg["data"])
        n = min(cfg["max_auctions"], traj.offsets.shape[0] - 1)
        table, off = traj.table[:n], np.asarray(traj.offsets[:n + 1], np.int64)
        rec = dict(calls=np.asarray(traj.calls[:off[-1]], np.uint8), offsets=off, board=None, dealer=None, vul=None,
                   seat_nets=np.zeros((n, 4), np.int32))
    else:
        table = load_table(cfg["deals"]) if cfg["deals"] else synthetic_deal_table(max(cfg["boards"], 1000), seed=0)
        rec = posterior.selfplay_auctions(nets[0], nets[1 % len(nets)], table, cfg["boards"], seed=cfg["seed"], device=dev)
    report = posterior.hand_reading(nets[:2], table, rec["calls"], rec["offsets"], rec["seat_nets"], board=rec["board"],
                                    dealer=rec["dealer"], vul=rec["vul"], at=cfg["at"], **kw)
    report = dict(config=cfg, by_observer_net=report)
    with open(cfg["out"], "w") as fh:
        json.dump(report, fh, indent=1)
    print(json.dumps(report["by_observer_net"], indent=1))


if __name__ == "__main__":
    main(sys.argv[1:])
