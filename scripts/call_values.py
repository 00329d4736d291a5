"""Which calls of some nets cost IMPs, and what they should have called instead (DESIGN.md f16).

    python scripts/call_values.py nets=model-sl.pkl,model-rl.pkl [deals=dds_results/test_000.npy] num_eval_envs=1000 \
        [opponent=-1] [top=20] [min_count=30] [out=call_values.json]
    python scripts/call_values.py models_directory=models exp_name=run skip_interval=100 max_step=10000 ...
    python -m torch.distributed.run --nproc-per-node N scripts/call_values.py nets=...

The nets of `nets=` (comma-separated .pkl paths), or a run's checkpoints chosen as scripts/selfplay_league.py chooses them.
Each net plays all four seats of num_eval_envs boards of the deal table `deals=` (synthetic when omitted; rng PRNGKey(0)),
or with opponent=k plays against net k, and every legal alternative of every decision is played out
(evaluation.make_call_values_evaluate).  Writes a JSON report: per net its mean regret, regret by context and top
deviations (call_values.CallValues.summary) and its comparison with the first net (call_values.compare).
"""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, call_values, random as brandom  # noqa: E402
from brl_b200.deals import load_table  # noqa: E402
from brl_b200.evaluation import list_league_checkpoints, make_call_values_evaluate  # noqa: E402
from brl_b200.models import load_params  # noqa: E402

DEFAULTS = dict(nets="", models_directory="models", exp_name="", skip_interval=100, max_step=10000, deals="",
                num_eval_envs=1000, opponent=-1, activation="relu", model_type="DeepMind", out="call_values.json",
                max_envs=1 << 20, top=20, min_count=30)


def parse_args(argv):
    cfg = dict(DEFAULTS)
    for arg in argv:
        key, sep, value = arg.partition("=")
        if not sep or key not in cfg:
            raise SystemExit(f"expected key=value with key in {sorted(cfg)}, got {arg!r}")
        cfg[key] = type(DEFAULTS[key])(value)
    if not (cfg["nets"] or cfg["exp_name"]):
        raise SystemExit("name the nets: nets=a.pkl,b.pkl, or exp_name= (a run's checkpoints)")
    return cfg


def net_paths(cfg):
    if cfg["nets"]:
        return [p for p in cfg["nets"].split(",") if p]
    names = list_league_checkpoints(cfg["models_directory"], cfg["exp_name"], cfg["skip_interval"], cfg["max_step"])
    return [os.path.join(cfg["models_directory"], cfg["exp_name"], name) for name in names]


def main(argv=None):
    cfg = parse_args(sys.argv[1:] if argv is None else argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    paths = net_paths(cfg)
    env = BridgeBidding(table=load_table(cfg["deals"]) if cfg["deals"] else None, device=dev)
    evaluate = make_call_values_evaluate(env, cfg["activation"], cfg["model_type"], cfg["num_eval_envs"],
                                         max_envs=cfg["max_envs"])
    result = evaluate([load_params(p, dev) for p in paths], brandom.PRNGKey(0),
                      opponent=None if cfg["opponent"] < 0 else cfg["opponent"])
    if world == 1 or dist.get_rank() == 0:
        nets = call_values.from_sums(result)
        names = [os.path.basename(p) for p in paths]
        report = {name: dict(values=v.summary(cfg["top"], cfg["min_count"]), versus_first=call_values.compare(nets[0], v))
                  for name, v in zip(names, nets)}
        with open(cfg["out"], "w") as fh:
            json.dump(dict(nets=names, num_eval_envs=cfg["num_eval_envs"], opponent=cfg["opponent"], report=report), fh,
                      indent=1)
        for name, v in zip(names, nets):
            print(f"{name}: {v.decisions} decisions, mean regret {v.mean_regret():.3f} IMPs")
        print(json.dumps({"nets": len(names), "out": cfg["out"]}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
