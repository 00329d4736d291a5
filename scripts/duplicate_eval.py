"""eval.py: a duplicate match of two saved models, played as one device-resident call (brl_duplicate_match).

    python scripts/duplicate_eval.py team1_model_path=bridge_models/model-sl.pkl team2_model_path=bridge_models/model-pretrained-rl.pkl \
        [team1_activation=relu] [team1_model_type=DeepMind] [team2_activation=relu] [team2_model_type=DeepMind] \
        [num_eval_envs=100] [eval_dds=dds_results/test_000.npy]
    python -m torch.distributed.run --nproc-per-node N scripts/duplicate_eval.py ...   (num_eval_envs is the whole match)

The arguments are EVALConfig's keys as key=value.  As in eval.py the boards come from rng PRNGKey(0), team 1 sits on
players 0/1 and the script prints `IMP: mean ± SE`.  The whole match runs through
evaluation.make_device_duplicate_evaluate: init, the bidding loop and the statistics stay on the GPU.  Both teams must
be the same architecture (the device loop forwards a pool of nets of one kind), which every bundled model is.
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, dist as bdist, random as brandom  # noqa: E402
from brl_b200.evaluation import make_device_duplicate_evaluate  # noqa: E402
from brl_b200.models import load_params  # noqa: E402

DEFAULTS = dict(team1_model_path="", team2_model_path="", team1_activation="relu", team1_model_type="DeepMind",
                team2_activation="relu", team2_model_type="DeepMind", num_eval_envs=100,
                eval_dds="dds_results/test_000.npy")


def parse_args(argv):
    cfg = dict(DEFAULTS)
    for arg in argv:
        key, sep, value = arg.partition("=")
        if not sep or key not in cfg:
            raise SystemExit(f"expected key=value with key in {sorted(cfg)}, got {arg!r}")
        cfg[key] = type(DEFAULTS[key])(value)
    if not cfg["team1_model_path"] or not cfg["team2_model_path"]:
        raise SystemExit("team1_model_path and team2_model_path are required")
    if (cfg["team1_activation"], cfg["team1_model_type"]) != (cfg["team2_activation"], cfg["team2_model_type"]):
        raise SystemExit("the device-loop match needs both teams to be the same architecture (activation and model_type)")
    if cfg["num_eval_envs"] <= 0:
        raise SystemExit("num_eval_envs must be > 0")
    return cfg


def main(argv=None):
    cfg = parse_args(sys.argv[1:] if argv is None else argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rank, world = bdist.rank_world()
    lo, hi = bdist.shard_range(cfg["num_eval_envs"], rank, world)
    env = BridgeBidding(cfg["eval_dds"], device=dev)
    duplicate_evaluate = make_device_duplicate_evaluate(env, cfg["team1_activation"], cfg["team1_model_type"], hi - lo,
                                                        env_offset=lo)
    print(f"num envs: {cfg['num_eval_envs']}")
    team1_params = load_params(cfg["team1_model_path"], dev)
    team2_params = load_params(cfg["team2_model_path"], dev)
    print("---------------------------------------------------")
    print(f"{cfg['team1_model_path']} vs. {cfg['team2_model_path']}")
    log, _, _, _ = duplicate_evaluate(team1_params, team2_params, brandom.PRNGKey(0))
    if rank == 0:
        print(f"IMP: {float(log[0])} ± {float(log[1])}")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
