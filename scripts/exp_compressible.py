"""Does compressible device memory speed up the bench rollout?  Plain (torch) against compressible
(brl_alloc_compressible) observation / mask trajectories, one process, A/B alternated inside every round.

For each shape (bench: 8192 envs x 32 steps; bench.py --sweep: 65,536 x 8 and 1,048,576 x 2) and writer count it
times `rollout_random` into each trajectory with CUDA events (median / min / max over rounds), and checks that both
trajectories receive bit-identical outputs (all six streams and the statistics) from the same start state.  Also
records the card, its power limit, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, the allocation granularity and
whether the driver granted compression.

    python scripts/exp_compressible.py [out.json]
"""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import _lib, ops  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402

DEV = "cuda:0"
SEED = 20241017  # bench.py
CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = 107  # cuda.h


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def compression_attribute():
    cu = C.CDLL("libcuda.so.1")
    dev, v = C.c_int(0), C.c_int(-1)
    assert cu.cuDeviceGet(C.byref(dev), 0) == 0
    assert cu.cuDeviceGetAttribute(C.byref(v), CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev) == 0
    return v.value


def trajectories(n, k):
    """(plain, compressible) EnvOutputs of [k, n, ...] rows; rewards / terminated / player stay torch in both"""
    comp = ops.EnvOutputs(n, DEV, rows=k)
    plain = ops.EnvOutputs(n, DEV, rows=k)
    plain.observation = torch.empty_like(comp.observation)
    plain.legal_action_mask = torch.empty_like(comp.legal_action_mask)
    return plain, comp


def run_shape(table, n, k, writers, rounds, reps):
    state0, out0 = ops.new_state(n, DEV), ops.EnvOutputs(n, DEV)
    ops.init(ops.make_keys(SEED, n, DEV), table, state0, out0)
    bufs = dict(zip(("plain", "compressible"), trajectories(n, k)))
    # bit-exactness: same start state, same seed, default launch shape, then every writer count
    ref, identical = None, True
    for name, traj in bufs.items():
        for w in (0,) + tuple(writers):
            st = state0.clone()
            act = torch.empty((k, n), dtype=torch.int32, device=DEV)
            stats = torch.zeros(4, dtype=torch.int64, device=DEV)
            ops.rollout_random(st, table, k, traj, seed=SEED, step0=0, action_out=act, stats=stats, tune=_lib.tune(writers=w))
            torch.cuda.synchronize()
            got = (traj.observation, traj.legal_action_mask, traj.rewards, traj.terminated, traj.current_player, act, stats, st)
            if ref is None:
                ref = [t.clone() for t in got]
            else:
                identical &= all(torch.equal(a, b) for a, b in zip(ref, got))
    del ref
    state = state0.clone()
    res = {(name, w): [] for w in writers for name in bufs}
    step = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for w in writers:
            for name, traj in bufs.items():
                tune = _lib.tune(writers=w)
                for _ in range(3):
                    ops.rollout_random(state, table, k, traj, seed=SEED, step0=step, tune=tune); step += k
                torch.cuda.synchronize()
                e0.record()
                for _ in range(reps):
                    ops.rollout_random(state, table, k, traj, seed=SEED, step0=step, tune=tune); step += k
                e1.record()
                torch.cuda.synchronize()
                res[(name, w)].append(1e3 * e0.elapsed_time(e1) / reps)
    rows = []
    for (name, w), v in res.items():
        rows.append({"n_envs": n, "sub_steps": k, "writers": w, "memory": name, "median_us": round(statistics.median(v), 2),
                     "min_us": round(min(v), 2), "max_us": round(max(v), 2), "rounds": rounds, "launches_per_round": reps,
                     "env_steps_per_s": n * k / (statistics.median(v) * 1e-6)})
    rows.sort(key=lambda r: r["median_us"])
    return {"n_envs": n, "sub_steps": k, "bit_identical": identical, "results": rows}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    L = _lib.load()
    table = torch.as_tensor(synthetic_deal_table(100_000, 0), device=DEV)
    probe = _lib.CompressibleBuffer(1 << 20, 0)
    info = {"card": card(), "generic_compression_supported": compression_attribute(),
            "granularity_bytes": int(L.brl_compressible_granularity(0)), "compression_granted": probe.granted}
    del probe
    print(json.dumps(info), flush=True)
    report = {"info": info, "shapes": []}
    for n, k, writers, rounds, reps in ((8192, 32, (3, 4, 5, 6, 7), 15, 40), (65536, 8, (3, 4, 5), 9, 20),
                                        (1048576, 2, (3, 4, 5), 7, 10)):
        r = run_shape(table, n, k, writers, rounds, reps)
        report["shapes"].append(r)
        print(f"n={n} k={k} bit_identical={r['bit_identical']}")
        for row in r["results"]:
            print(f"  w{row['writers']} {row['memory']:12s} median {row['median_us']:9.2f} us  min {row['min_us']:9.2f}  "
                  f"max {row['max_us']:9.2f}  {row['env_steps_per_s']:.3e} env-steps/s", flush=True)
        torch.cuda.empty_cache()
    info["card_after"] = card()
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
