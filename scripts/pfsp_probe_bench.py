"""The PFSP probe over the model zoo: one make_device_duplicate_evaluate call per zoo model (the zoo as host NumPy dicts, each
model copied to the device and packed for its match) against make_device_pfsp_probe (the zoo packed in HBM, one
brl_duplicate_match call for the whole zoo); then one whole PFSP iteration of ppo.train with each zoo.

    python scripts/pfsp_probe_bench.py [--reps 5] [--train-zoo 100] [--out profiles/r06_pfsp_probe_b200.json]

Probe legs: K zoo models at num_prioritized_envs = 100 boards for K = 10, 100, 400, K = 100 at 1,000 boards, and K = 10 in a
zoo of capacity 400 (ppo.train allocates the zoo for the whole run, so while it fills the probe plays over M = 1 + capacity
nets).  Every
timed call is a whole probe, from the learner's parameters to the K statistics on the host, on the host clock around work
that ends in a device synchronise.  After one untimed call of each (its time and the new graph builds are recorded apart:
the one-time capture / instantiate cost when K changes) the two probes alternate call by call, and every pair must give
the same statistics.  The zoo models are seeded nets with a trained net's logit scale (policy head x 128), drawn on the device.

ppo.train leg: ppo.py's shape (8192 envs x 32 steps, minibatch 1024, 10 epochs), prioritized_fictitious
with ratio_model_zoo = 1 and a save every iteration, run for --train-zoo + 1 iterations so that the last iterations draw
from a zoo of about --train-zoo models; the host zoo run has the device zoo refused up front.  Per-iteration time is the
host clock between log_fn calls; with the device zoo each probe call inside the run is timed as
well, and ppo.train's own time/* entries are kept per iteration.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import BridgeBidding, ops, ppo, random as brandom  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200.evaluation import make_device_duplicate_evaluate, make_device_pfsp_probe  # noqa: E402
from brl_b200.models import LAYERS, SIZES  # noqa: E402
from brl_b200.zoo import ModelZoo  # noqa: E402


def device_net(seed, dev):
    """haiku-like init drawn on the device (normal clipped to +-2, / sqrt(fan_in)), policy head x 128"""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    p = {}
    for name, (fi, fo) in zip(LAYERS, SIZES):
        w = torch.randn((fi, fo), generator=g, device=dev).clamp_(-2, 2) / float(np.sqrt(fi))
        p[name] = {"w": w * 128 if name == LAYERS[4] else w, "b": torch.zeros(fo, device=dev)}
    return p


def sync_time(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def probe_leg(env, current, host_zoo, zoo, n, reps, key, dev):
    K = len(zoo)
    per_model = make_device_duplicate_evaluate(env, "relu", "DeepMind", n)
    probe = make_device_pfsp_probe(env, "relu", "DeepMind", n)

    def old():   # ppo.train's probe with the host zoo: zoo_model(k) (H2D) + pack + one match per model
        return [per_model(current, {name: {kk: torch.as_tensor(v, device=dev) for kk, v in m[name].items()} for name in LAYERS},
                          key)[0] for m in host_zoo]

    def new():
        return probe(current, zoo, key)

    row = {"K": K, "capacity": zoo.capacity, "boards": n}
    for name, fn in (("per_model", old), ("one_call", new)):
        b0 = ops.duplicate_match_graph_builds()
        row[f"{name}_first_call_ms"], _ = sync_time(fn)
        row[f"{name}_graph_builds_first_call"] = ops.duplicate_match_graph_builds() - b0
    b0 = ops.duplicate_match_graph_builds()
    t_old, t_new = [], []
    for _ in range(reps):
        to, so = sync_time(old)
        tn, sn = sync_time(new)
        if [tuple(s) for s in so] != [tuple(s) for s in sn]:
            raise SystemExit(f"K={K} n={n}: the one-call probe and the per-model matches differ")
        t_old.append(to)
        t_new.append(tn)
    row["graph_builds_warm"] = ops.duplicate_match_graph_builds() - b0
    med = lambda v: float(np.median(v))  # noqa: E731
    row.update(per_model_ms=t_old, one_call_ms=t_new, per_model_median_ms=med(t_old), one_call_median_ms=med(t_new),
               speedup=med(t_old) / med(t_new), equal_statistics=True,
               live_rows_per_model=n, grouped_rows_per_model=ops.model_rows_capacity(n * K, 1 + K) // (1 + K))
    print(json.dumps({k: v for k, v in row.items() if not k.endswith("_ms") or "median" in k or "first" in k}), flush=True)
    return row


def train_leg(device_zoo, zoo_size, dev):
    """per-iteration times, and with the device zoo each probe call's time (it ends in its host read of the statistics)"""
    it_times, probe_ms = [], []
    orig_fits, orig_probe = ppo.device_zoo_fits, ppo.make_device_pfsp_probe
    if not device_zoo:
        ppo.device_zoo_fits = lambda *a, **kw: False

    def timed_probe(*a, **kw):
        probe = orig_probe(*a, **kw)

        def call(*pa, **pkw):
            t, out = sync_time(lambda: probe(*pa, **pkw))
            probe_ms.append(t)
            return out
        call.reserve = probe.reserve
        return call
    ppo.make_device_pfsp_probe = timed_probe
    last = [None]

    def log_fn(log):
        now = time.perf_counter()
        if last[0] is not None:
            it_times.append((now - last[0]) * 1e3)
        last[0] = now

    config = dict(num_envs=8192, num_steps=32, minibatch_size=1024, total_timesteps=8192 * 32 * (zoo_size + 1),
                  self_play=True, ratio_model_zoo=1.0, prioritized_fictitious=True, num_model_zoo=zoo_size,
                  save_model_interval=1, save_model=False)
    try:
        _, logs = ppo.train(config, brandom.PRNGKey(0), tables=[synthetic_deal_table(100_000, seed=k) for k in range(2)],
                            eval_table=synthetic_deal_table(10_000, seed=9), device=dev, log_fn=log_fn)
    finally:
        ppo.device_zoo_fits, ppo.make_device_pfsp_probe = orig_fits, orig_probe
    return it_times, probe_ms, logs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--train-zoo", type=int, default=100)
    ap.add_argument("--out", default="profiles/r06_pfsp_probe_b200.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    env = BridgeBidding(table=synthetic_deal_table(10_000, seed=1), device=dev)
    key = brandom.PRNGKey(0)
    current = device_net(1, dev)
    legs = ((10, 10, 100), (100, 100, 100), (400, 400, 100), (100, 100, 1000), (10, 400, 100))   # (K, capacity, boards)
    zoos = {(K, cap): ModelZoo(cap, dev) for K, cap, _ in legs}
    host_zoo = []
    for k in range(max(K for K, _, _ in legs)):
        net = device_net(1000 + k, dev)
        host_zoo.append(ppo.params_to_host(net))
        for (K, _), z in zoos.items():
            if k < K:
                z.append(net)
    del net
    rows = []
    for K, cap, n in legs:
        rows.append(probe_leg(env, current, host_zoo[:K], zoos[K, cap], n, args.reps, key, dev))
    del zoos, host_zoo
    torch.cuda.empty_cache()
    result = {"card": card, "reps": args.reps,
              "timing": "host clock around whole probes ending in a device synchronise; per-model and one-call probes "
                        "alternating after one untimed first call of each",
              "probe_rows": rows}
    write(args.out, result)   # the probe legs stand on their own

    train = {}
    tail = 5
    for name, device_zoo in (("host_zoo", False), ("device_zoo", True)):
        it_times, probe_ms, logs = train_leg(device_zoo, args.train_zoo, dev)
        train[name] = {"iteration_ms": it_times, f"last_{tail}_median_ms": float(np.median(it_times[-tail:])),
                       "logs": logs, **{k.replace("time/", "") + "_ms": [1e3 * log[k] for log in logs[1:]]
                                        for k in ("time/eval", "time/rollout", "time/calc_gae", "time/update")}}
        if probe_ms:
            train[name].update(probe_ms=probe_ms, **{f"probe_last_{tail}_median_ms": float(np.median(probe_ms[-tail:]))})
        print(json.dumps({name: train[name][f"last_{tail}_median_ms"]}), flush=True)
        torch.cuda.empty_cache()
    host_logs, dev_logs = train["host_zoo"].pop("logs"), train["device_zoo"].pop("logs")
    same = all(np.isclose(d[k], h[k], rtol=1e-12, atol=0) for h, d in zip(host_logs, dev_logs)
               for k in h if k.startswith(("train/", "eval/")))
    result["ppo_train"] = {"shape": "8192 envs x 32 steps, minibatch 1024, update_epochs 10, num_prioritized_envs 100, "
                                    f"prioritized_fictitious, zoo of up to {args.train_zoo} models (one save per iteration)",
                           "timing": "host clock between log_fn calls; the last iterations draw from the fullest zoo",
                           "logs_equal": bool(same), **train}
    write(args.out, result)


def write(path, result):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"card": result["card"], "out": path}), flush=True)


if __name__ == "__main__":
    main()
