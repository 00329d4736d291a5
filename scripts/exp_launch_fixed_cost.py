"""Fixed per-launch cost of the bench rollout kernel: time back-to-back `brl_rollout_random` launches at 8192 envs for
k = 1 .. 64 steps and fit t(k) = a + b * k.  The intercept a is what one launch costs beyond its k env steps: the
prologue (state load, deal-table gathers), the phase in which only the env warp works, the last phase in which only
the writers work, and the gap between launches.

    python scripts/exp_launch_fixed_cost.py [--rounds R] [--reps N] [--out file.json]
    BRL_B200_LIB=brl_b200/lib/libbrl_roletiming.so python scripts/exp_launch_fixed_cost.py --role
        (library built by `python scripts/build_variant.py roletiming -DBRL_ROLE_TIMING`): SM clocks per block of the
        prologue, of phase 0 and of the last phase, by role, at 8192 envs x 32 steps."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import _lib, ops  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402

N = 8192
KS = (1, 2, 4, 8, 16, 32, 64)


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except Exception as exc:  # the measurement stands without it, but says so
        return {"error": str(exc)}


def setup(dev, table, k):
    state, out0 = ops.new_state(N, dev), ops.EnvOutputs(N, dev)
    ops.init(ops.make_keys(1, N, dev), table, state, out0)
    return state, ops.EnvOutputs(N, dev, rows=k)


def sweep(args, dev, table):
    runs = {k: setup(dev, table, k) for k in KS}
    step = {k: 0 for k in KS}

    def launches(k, count):
        state, traj = runs[k]
        for _ in range(count):
            ops.rollout_random(state, table, k, traj, seed=1, step0=step[k])
            step[k] += k

    for k in KS:  # warm-up: module load, first touch of every trajectory
        launches(k, 3)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per_round = {k: [] for k in KS}
    for _ in range(args.rounds):
        for k in KS:
            e0.record()
            launches(k, args.reps)
            e1.record()
            torch.cuda.synchronize()
            per_round[k].append(1e3 * e0.elapsed_time(e1) / args.reps)
    med = np.array([np.median(per_round[k]) for k in KS])
    b, a = np.polyfit(np.array(KS, dtype=float), med, 1)
    fit = {"a_us": a, "b_us_per_step": b,
           "residual_us": {str(k): float(m - (a + b * k)) for k, m in zip(KS, med)}}
    # the bench shape sits at k = 32; the short launches weigh the same in the fit as the long ones
    b2, a2 = np.polyfit(np.array(KS[2:], dtype=float), med[2:], 1)
    fit_k4 = {"a_us": a2, "b_us_per_step": b2, "ks": list(KS[2:])}
    return {"n": N, "ks": list(KS), "rounds": args.rounds, "reps_per_round": args.reps,
            "us_per_launch_median": {str(k): float(m) for k, m in zip(KS, med)},
            "us_per_launch_min_max": {str(k): [min(per_round[k]), max(per_round[k])] for k in KS},
            "fit": fit, "fit_k_ge_4": fit_k4}


def role(dev, table):
    L = _lib.load()
    L.brl_debug_role_phase_cycles.argtypes = [C.c_void_p, C.c_int]
    L.brl_debug_role_cycles.argtypes = [C.c_void_p, C.c_int]
    k, reps = 32, 10
    state, traj = setup(dev, table, k)
    for i in range(3):
        ops.rollout_random(state, table, k, traj, seed=1, step0=i * k)
    torch.cuda.synchronize()
    ph, tot = (C.c_ulonglong * 16)(), (C.c_ulonglong * 8)()
    L.brl_debug_role_phase_cycles(ph, 1)
    L.brl_debug_role_cycles(tot, 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        ops.rollout_random(state, table, k, traj, seed=1, step0=(3 + i) * k)
    e1.record()
    torch.cuda.synchronize()
    L.brl_debug_role_phase_cycles(ph, 1)
    L.brl_debug_role_cycles(tot, 1)
    blocks = 296  # balanced grid at 8192 envs: 2 blocks per SM
    per_block = lambda v: v / (reps * blocks)  # noqa: E731
    names = ["env_work", "env_barrier", "warp0_work", "warp0_barrier", "other_writers_work_sum", "other_writers_barrier_sum"]
    return {"n": N, "k": k, "us_per_launch_timing_build": 1e3 * e0.elapsed_time(e1) / reps,
            "sm_clocks_per_block": {
                "prologue": {"env_warp": per_block(ph[6]), "warp0": per_block(ph[7])},
                "phase0": {nm: per_block(ph[j]) for j, nm in enumerate(names)},
                "last_phase": {nm: per_block(ph[8 + j]) for j, nm in enumerate(names)},
                "mean_phase_all": {nm: per_block(tot[j]) / (k + 1) for j, nm in enumerate(names)}}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=12)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--role", action="store_true")
    ap.add_argument("--label", default="")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = "cuda:0"
    table = torch.as_tensor(synthetic_deal_table(100000, 0), device=dev)
    res = {"label": args.label, "gpu": gpu_info(), "torch": torch.__version__}
    res.update(role(dev, table) if args.role else sweep(args, dev, table))
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
