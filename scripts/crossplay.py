"""Cross-play over the saved checkpoints of one training run: how well every two of its nets bid together as partners.

    python scripts/crossplay.py models_directory=models exp_name=pbt-run opp_model_path=model-sl.pkl num_eval_envs=100 \
        skip_interval=100 max_step=10000 [partner_opp_model_path=...] [eval_dds=dds_results/test_000.npy] [out_dir=.]
    python -m torch.distributed.run --nproc-per-node N scripts/crossplay.py exp_name=...

Checkpoints are chosen as scripts/selfplay_league.py chooses them (evaluation.list_league_checkpoints).  Every ordered
partnership (a, b) of the M checkpoints -- a on player 0, b on player 1, the diagonal included -- plays one duplicate match
over the same num_eval_envs boards (rng PRNGKey(0)) against the fixed pair (opp_model_path, partner_opp_model_path; the
second defaults to the first), all M^2 matches batched on the GPU with each chunk of up to max_envs envs per rank played as
one brl_duplicate_match call (evaluation.make_crossplay_evaluate).

Writes crossplay_{exp_name}.npy (imp[a, b], the mean IMP of partnership (a, b)) and crossplay_{exp_name}.npz with imp, se,
win_rate and the checkpoint list.
"""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, random as brandom  # noqa: E402
from brl_b200.evaluation import list_league_checkpoints, make_crossplay_evaluate  # noqa: E402
from brl_b200.models import load_params  # noqa: E402

DEFAULTS = dict(models_directory="models", exp_name="pretrained-rl-with-sp", opp_model_path="", partner_opp_model_path="",
                num_eval_envs=100, skip_interval=100, max_step=10000, activation="relu", model_type="DeepMind",
                eval_dds="dds_results/test_000.npy", out_dir=".", max_envs=1 << 20)


def parse_args(argv):
    cfg = dict(DEFAULTS)
    for arg in argv:
        key, sep, value = arg.partition("=")
        if not sep or key not in cfg:
            raise SystemExit(f"expected key=value with key in {sorted(cfg)}, got {arg!r}")
        cfg[key] = type(DEFAULTS[key])(value)
    if not cfg["opp_model_path"]:
        raise SystemExit("opp_model_path= names the opponents' net")
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
    if not names:
        raise SystemExit("cross-play needs at least one checkpoint")
    params_list = [load_params(os.path.join(cfg["models_directory"], cfg["exp_name"], name), dev) for name in names]
    opp = load_params(cfg["opp_model_path"], dev)
    opp_partner = load_params(cfg["partner_opp_model_path"], dev) if cfg["partner_opp_model_path"] else opp
    env = BridgeBidding(cfg["eval_dds"], device=dev)
    crossplay = make_crossplay_evaluate(env, cfg["activation"], cfg["model_type"], cfg["num_eval_envs"],
                                        max_envs=cfg["max_envs"])
    stats, imp = crossplay(params_list, (opp, opp_partner), brandom.PRNGKey(0))
    if world == 1 or dist.get_rank() == 0:
        M = len(names)
        se, win_rate = np.full((M, M), np.nan), np.full((M, M), np.nan)
        for (a, b), (_, s, w) in stats.items():
            se[a, b], win_rate[a, b] = s, w
        base = os.path.join(cfg["out_dir"], f"crossplay_{cfg['exp_name']}")
        with open(base + ".npy", "wb") as fh:
            np.save(fh, imp)
        np.savez(base + ".npz", imp=imp, se=se, win_rate=win_rate, checkpoints=np.asarray(names))
        print(json.dumps({"checkpoints": M, "matches": len(stats), "boards": len(stats) * cfg["num_eval_envs"],
                          "out": base + ".npz"}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
