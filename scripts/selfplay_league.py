"""workspace/eval_selfplay_league.py: a duplicate match between every pair of saved checkpoints of one training run.

    python scripts/selfplay_league.py models_directory=models exp_name=pretrained-rl-with-sp num_eval_envs=100 \
        skip_interval=100 max_step=10000 [eval_dds=dds_results/test_000.npy] [out_dir=.] [max_envs=1048576]
    python -m torch.distributed.run --nproc-per-node N scripts/selfplay_league.py exp_name=...

The arguments are the script's config keys as key=value (SelfplayLeagueConfig).  Checkpoints are the files of
models_directory/exp_name with "params" in the name, step % skip_interval == 0 and step <= max_step, sorted; ppo.train's
params-XXXXXXXX.pkl qualify, its opt_state-*.pkl do not.  Every pair (i, j), i < j, plays one
make_simple_duplicate_evaluate match over the same num_eval_envs boards (rng PRNGKey(0)), all matches batched on the GPU
with each chunk of up to max_envs envs per rank played as one device-resident brl_duplicate_match call
(evaluation.make_selfplay_league_evaluate).

Writes win_lose_{exp_name}.npy (the reference's output) and win_lose_{exp_name}.npz with win_lose, win_lose_dis,
win_lose_clip, the per-pair imp / se / win_rate matrices (entry [i, j] = the match with team 1 = i, team 2 = j) and the
checkpoint list.  The reference's heatmaps (seaborn / matplotlib) are not drawn: neither library is a dependency here.
save_fig_directory_path is accepted and ignored.
"""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, random as brandom  # noqa: E402
from brl_b200.evaluation import list_league_checkpoints, make_selfplay_league_evaluate  # noqa: E402
from brl_b200.models import load_params  # noqa: E402

DEFAULTS = dict(models_directory="models", exp_name="pretrained-rl-with-sp", num_eval_envs=100, skip_interval=100,
                max_step=10000, save_fig_directory_path="", activation="relu", model_type="DeepMind",
                eval_dds="dds_results/test_000.npy", out_dir=".", max_envs=1 << 20)


def parse_args(argv):
    cfg = dict(DEFAULTS)
    for arg in argv:
        key, sep, value = arg.partition("=")
        if not sep or key not in cfg:
            raise SystemExit(f"expected key=value with key in {sorted(cfg)}, got {arg!r}")
        cfg[key] = type(DEFAULTS[key])(value)
    return cfg


def main(argv=None):
    cfg = parse_args(sys.argv[1:] if argv is None else argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    names = list_league_checkpoints(cfg["models_directory"], cfg["exp_name"], cfg["skip_interval"], cfg["max_step"])
    print(names)
    if len(names) < 2:
        raise SystemExit("a league needs at least two checkpoints")
    params_list = [load_params(os.path.join(cfg["models_directory"], cfg["exp_name"], name), dev) for name in names]
    env = BridgeBidding(cfg["eval_dds"], device=dev)
    league = make_selfplay_league_evaluate(env, cfg["activation"], cfg["model_type"], cfg["num_eval_envs"],
                                           max_envs=cfg["max_envs"])
    stats, win_lose, win_lose_dis, win_lose_clip = league(params_list, brandom.PRNGKey(0))
    if world == 1 or dist.get_rank() == 0:
        M = len(names)
        imp, se, win_rate = (np.full((M, M), np.nan) for _ in range(3))
        for (i, j), (m, s, w) in stats.items():
            imp[i, j], se[i, j], win_rate[i, j] = m, s, w
        base = os.path.join(cfg["out_dir"], f"win_lose_{cfg['exp_name']}")
        with open(base + ".npy", "wb") as fh:
            np.save(fh, win_lose)
        np.savez(base + ".npz", win_lose=win_lose, win_lose_dis=win_lose_dis, win_lose_clip=win_lose_clip, imp=imp, se=se,
                 win_rate=win_rate, checkpoints=np.asarray(names))
        print(json.dumps({"checkpoints": M, "matches": len(stats), "boards": len(stats) * cfg["num_eval_envs"],
                          "out": base + ".npz"}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
