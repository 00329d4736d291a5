"""What the calls of some nets (and of a file of recorded auctions) promise: hand strength and shape per call, in the first
round of the auction (DESIGN.md f15).

    python scripts/bidding_system.py nets=model-sl.pkl,model-rl.pkl [data=test.txt] [deals=dds_results/test_000.npy] \
        num_eval_envs=10000 [opponent=-1] [out=bidding_system.json]
    python scripts/bidding_system.py models_directory=models exp_name=run skip_interval=100 max_step=10000 ...
    python -m torch.distributed.run --nproc-per-node N scripts/bidding_system.py nets=...

Sources: the nets of `nets=` (comma-separated .pkl paths), or a run's checkpoints chosen as scripts/selfplay_league.py
chooses them (evaluation.list_league_checkpoints), then the auctions of `data=` (an OpenSpiel data file, parsed and checked
as sl.train reads it).  Each net plays all four seats of num_eval_envs boards of the deal table `deals=` (synthetic when
omitted; rng PRNGKey(0)), both tables of each board (evaluation.make_bidding_system_evaluate); with opponent=k every net
plays against net k instead.

Writes a JSON report: per source its histogram summary (system.BiddingSystem.summary) and its comparison with the first
source (system.compare); prints each source's openings (OPEN(0..3)) and the responses to the one-level openings.
"""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, random as brandom, sl, system  # noqa: E402
from brl_b200.deals import load_table  # noqa: E402
from brl_b200.evaluation import list_league_checkpoints, make_bidding_system_evaluate  # noqa: E402
from brl_b200.models import load_params  # noqa: E402

DEFAULTS = dict(nets="", models_directory="models", exp_name="", skip_interval=100, max_step=10000, data="", deals="",
                num_eval_envs=10000, opponent=-1, activation="relu", model_type="DeepMind", out="bidding_system.json",
                max_envs=1 << 20)


def parse_args(argv):
    cfg = dict(DEFAULTS)
    for arg in argv:
        key, sep, value = arg.partition("=")
        if not sep or key not in cfg:
            raise SystemExit(f"expected key=value with key in {sorted(cfg)}, got {arg!r}")
        cfg[key] = type(DEFAULTS[key])(value)
    if not (cfg["nets"] or cfg["exp_name"] or cfg["data"]):
        raise SystemExit("name the sources: nets=a.pkl,b.pkl, or exp_name= (a run's checkpoints), and / or data=")
    return cfg


def net_paths(cfg):
    if cfg["nets"]:
        return [p for p in cfg["nets"].split(",") if p]
    if cfg["exp_name"]:
        names = list_league_checkpoints(cfg["models_directory"], cfg["exp_name"], cfg["skip_interval"], cfg["max_step"])
        return [os.path.join(cfg["models_directory"], cfg["exp_name"], name) for name in names]
    return []


def first_round(name: str, s: system.BiddingSystem) -> str:
    """the openings by position and the responses to the one-level openings, as text"""
    lines = [f"== {name}"]
    for p in range(4):
        lines.append(f"-- {system.context_name(p)}: {int(s.decisions[p])} decisions")
        lines.extend("   " + r for r in s.describe(p, min_share=0.005))
    for bid in range(5):
        c = system.response_context(bid)
        if s.decisions[c]:
            lines.append(f"-- {system.context_name(c)}: {int(s.decisions[c])} decisions")
            lines.extend("   " + r for r in s.describe(c, min_share=0.005))
    return "\n".join(lines)


def main(argv=None):
    cfg = parse_args(sys.argv[1:] if argv is None else argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sources = {}
    paths = net_paths(cfg)
    if paths:
        env = BridgeBidding(table=load_table(cfg["deals"]) if cfg["deals"] else None, device=dev)
        evaluate = make_bidding_system_evaluate(env, cfg["activation"], cfg["model_type"], cfg["num_eval_envs"],
                                                max_envs=cfg["max_envs"])
        params_list = [load_params(p, dev) for p in paths]
        hist = evaluate(params_list, brandom.PRNGKey(0), opponent=None if cfg["opponent"] < 0 else cfg["opponent"])
        sources.update((os.path.basename(p), system.BiddingSystem(hist[m])) for m, p in enumerate(paths))
    if cfg["data"]:
        traj = sl.parse_trajectories(cfg["data"])
        sl.check_trajectories(traj, dev, cfg["data"])
        sources[os.path.basename(cfg["data"])] = system.from_auctions(traj, dev)
    if world == 1 or dist.get_rank() == 0:
        names = list(sources)
        first = sources[names[0]]
        report = {name: dict(system=s.summary(), versus_first=system.compare(first, s)) for name, s in sources.items()}
        with open(cfg["out"], "w") as fh:
            json.dump(dict(sources=names, first=names[0], num_eval_envs=cfg["num_eval_envs"], report=report), fh, indent=1)
        for name, s in sources.items():
            print(first_round(name, s))
        print(json.dumps({"sources": len(names), "out": cfg["out"]}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
