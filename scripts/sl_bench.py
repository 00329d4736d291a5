"""Timings of the supervised pre-training path on the GPU (brl_b200/sl.py), one JSON line on stdout:

  examples       brl_sl_examples, examples/s at B = 128 (sl.py's train_batch), 10,000 (its eval_batch) and 65,536, per
                 observation dtype (call positions drawn in-kernel)
  step           one SL optimizer step -- examples + brl_sl_grad + brl_mlp_adam_step -- at B = 128 and 1,024, with and
                 without the post-update accuracy forward (brl_sl_eval, sl.py:279)
  cpu_examples   the C oracle (oracle/sl_ref.replay_examples) building the same examples on all host cores: a reported
                 CPU comparison, not a tuned port (it steps the oracle env position group by position group from Python)

Device times are CUDA events around `iters` back-to-back calls after a warm-up.  The trajectories are 20,000 synthetic
random-legal auctions (~0.5 MB of calls and deal rows, L2-resident after the first call, as the training set of a real
run would largely be at these batch sizes); the outputs are rewritten in place on every call.

    python scripts/sl_bench.py [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def time_ms(fn, iters: int, warmup: int) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def gpu_info() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["nvidia_smi"] = out
    except Exception as exc:  # the card name from torch still identifies the measurement
        info["nvidia_smi"] = f"unavailable: {exc}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--no-cpu", action="store_true")
    args = ap.parse_args()
    from brl_b200 import ops
    from brl_b200.models import init_params
    from brl_b200.optim import flatten_params
    from oracle import sl_ref
    dev = torch.device("cuda:0")
    t = sl_ref.random_trajectories(20_000, seed=1)
    d = t.to(dev)
    rng = np.random.default_rng(0)
    res = {"gpu": gpu_info(), "n_trajectories": len(t), "mean_calls": float(np.diff(t.offsets).mean()),
           "iters": args.iters, "examples": {}, "step": {}, "cpu_examples": {}}
    for B in (128, 10_000, 65_536):
        traj = torch.as_tensor(rng.integers(0, len(t), B), dtype=torch.int32, device=dev)
        mask = torch.empty((B, 38), dtype=torch.uint8, device=dev)
        label = torch.empty(B, dtype=torch.int32, device=dev)
        for dt in (torch.uint8, torch.bfloat16, torch.float32):
            obs = torch.empty((B, 480), dtype=dt, device=dev)
            k = [0]

            def run():
                k[0] += 1
                ops.sl_examples(d["table"], d["calls"], d["offsets"], traj, obs, mask, label, seed=7, step=k[0])
            ms = time_ms(run, args.iters, args.warmup)
            res["examples"][f"B{B}_{str(dt).split('.')[-1]}"] = {"ms": ms, "examples_per_s": B / ms * 1e3}
    params = init_params(0, dev)
    flat, _ = flatten_params(params)
    blob = ops.mlp_pack_train(flat)
    m, v, grads = torch.zeros_like(flat), torch.zeros_like(flat), torch.empty_like(flat)
    acc_g, acc_e = ops.sl_acc(dev), ops.sl_acc(dev)
    for B in (128, 1024):
        scratch = ops.mlp_train_scratch(B, dev)
        traj = torch.as_tensor(rng.integers(0, len(t), B), dtype=torch.int32, device=dev)
        obs = torch.empty((B, 480), dtype=torch.uint8, device=dev)
        mask = torch.empty((B, 38), dtype=torch.uint8, device=dev)
        label = torch.empty(B, dtype=torch.int32, device=dev)
        stats = torch.zeros((2, 8), device=dev)
        for with_acc in (False, True):
            k = [0]

            def step():
                k[0] += 1
                ops.sl_examples(d["table"], d["calls"], d["offsets"], traj, obs, mask, label, seed=7, step=k[0])
                ops.sl_grad(obs, blob, scratch, mask, label, grads, stats[0], acc_g, ent_coef=0.0)
                ops.mlp_adam_step(flat, grads, m, v, acc_g[14:15], blob, step=k[0], lr=1e-6, eps=1e-8, max_grad_norm=0.0)
                if with_acc:
                    ops.sl_eval(obs, blob, scratch, mask, label, stats[1], acc_e)
            ms = time_ms(step, args.iters, args.warmup)
            res["step"][f"B{B}_{'with' if with_acc else 'without'}_train_accuracy"] = {"ms": ms, "examples_per_s": B / ms * 1e3}
        res["step"][f"B{B}_sl_grad_only"] = {"ms": time_ms(
            lambda: ops.sl_grad(obs, blob, scratch, mask, label, grads, stats[0], acc_g), args.iters, args.warmup)}
    if not args.no_cpu:
        threads = os.cpu_count() or 1
        res["cpu_examples"]["threads"] = threads
        for B in (10_000, 65_536):
            traj = rng.integers(0, len(t), B)
            pos = (rng.random(B) * np.diff(t.offsets)[traj]).astype(np.int64)
            t0 = time.perf_counter()
            sl_ref.replay_examples(t.table, t.calls, t.offsets, traj, pos, n_threads=threads)
            s = time.perf_counter() - t0
            res["cpu_examples"][f"B{B}"] = {"s": s, "examples_per_s": B / s}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
