"""K PPO learners on one GPU: K solo runs back to back against one population run, per update and per iteration.

    python scripts/population_bench.py [--ks 1 2 4 8] [--reps 3] [--iter-ks 1 2 4] [--iterations 4]
                                       [--out profiles/r11_population_b200.json]

One update is what ppo.train runs per iteration: update_epochs passes of num_minibatches optimizer steps over a
num_steps x num_envs rollout (defaults 10 x 256 steps of 1,024 samples over 32 x 8192).  Each learner has its own net,
its own synthetic rollout (sparse 0/1 bf16 observations as the tensor-core rollout records them, random legal masks,
actions, advantages) and its own lr / ent_coef / clip_eps.  For each K the two ways alternate in one process, each timed
with a host clock around work that ends in a device synchronise; the first pair is a warm-up and is also where the
learners' parameters of the two ways are compared for bit equality.  Besides the times the script records the device
memory a grouped update allocates per learner (its peak above what was allocated before it: rollouts, nets).

The iteration leg runs ppo.train K times and ppo.train_population once with the same K configs (ppo.train's defaults:
8192 envs x 32 steps, 10,000-env evaluations; different seeds, lr and ent_coef), alternating the two, and times each
iteration between consecutive log callbacks.  Iteration 0 (set-up effects, the every-10th duplicate evaluation) is left
out; the median of the others is reported.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from brl_b200 import ops, ppo  # noqa: E402
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from brl_b200 import random as brandom  # noqa: E402
from brl_b200.models import init_params, make_forward_pass  # noqa: E402
from brl_b200.optim import make_optimizer  # noqa: E402
from brl_b200.roll_out import Transition  # noqa: E402
from brl_b200.update import make_population_update_step, make_update_step  # noqa: E402

DEV = "cuda"


def _config(k, T, n, mbs, epochs):
    return dict(actor_illegal_action_mask=True, clip_eps=0.2 - 0.01 * k, ent_coef=0.01 * (k + 1), vf_coef=0.5,
                illegal_action_l2norm_coef=0.0, value_clipping=True, reward_scaling=False, num_minibatches=T * n // mbs,
                minibatch_size=mbs, update_epochs=epochs, num_steps=T, num_envs=n, total_timesteps=T * n * 100, num_updates=100,
                lr=3e-4 * (1 + k), anneal_lr=True, max_grad_norm=0.5, global_gradient_clipping=True,
                illegal_action_loss_stat="last", actor_model_type="DeepMind", actor_activation="relu")


def _rollout(seed, T, n):
    g = torch.Generator(device=DEV).manual_seed(seed)
    mask = torch.rand((T, n, 38), generator=g, device=DEV) < 0.5
    mask[..., 0] = True
    action = torch.multinomial(mask.reshape(-1, 38).float(), 1, generator=g)[:, 0].to(torch.int32).reshape(T, n)
    traj = Transition(done=torch.zeros((T, n), dtype=torch.bool, device=DEV), action=action,
                      value=torch.randn((T, n), generator=g, device=DEV) * 0.3, reward=torch.zeros((T, n), device=DEV),
                      log_prob=-torch.rand((T, n), generator=g, device=DEV) * 3,
                      obs=(torch.rand((T, n, 480), generator=g, device=DEV) < 0.04).to(torch.bfloat16), legal_action_mask=mask)
    return traj, torch.randn((T, n), generator=g, device=DEV), torch.randn((T, n), generator=g, device=DEV) * 0.3


def _gpu_label():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def bench_k(K, T, n, mbs, epochs, reps):
    fp = make_forward_pass("relu", "DeepMind", precision="tc")
    configs = [_config(k, T, n, mbs, epochs) for k in range(K)]
    rollouts = [_rollout(100 + k, T, n) for k in range(K)]
    params = [init_params(k, DEV) for k in range(K)]
    solo_steps = [(make_update_step(c, fp, o), o) for c, o in ((c, make_optimizer(c)) for c in configs)]
    pop_opts = [make_optimizer(c) for c in configs]
    pop_step = make_population_update_step(configs, fp, pop_opts)

    def runners(opts):
        return [(p, o.init(p), None, None, 0, brandom.PRNGKey(k)) for k, (p, o) in enumerate(zip(params, opts))]

    solo_runners = runners([o for _, o in solo_steps])
    pop_runners = runners(pop_opts)

    def run_solo():
        return [step(r, *ro) for (step, _), r, ro in zip(solo_steps, solo_runners, rollouts)]

    def run_pop():
        return pop_step(pop_runners, [r[0] for r in rollouts], [r[1] for r in rollouts], [r[2] for r in rollouts])

    a = run_solo()
    torch.cuda.synchronize()
    base_mem = torch.cuda.memory_allocated()  # the rollouts, nets and the solo outputs kept for the comparison below
    torch.cuda.reset_peak_memory_stats()
    b = run_pop()
    torch.cuda.synchronize()
    pop_peak = torch.cuda.max_memory_allocated() - base_mem
    equal = all(torch.equal(torch.cat([t.reshape(-1) for L in sa[0][0].values() for t in L.values()]).view(torch.int32),
                            torch.cat([t.reshape(-1) for L in sb[0][0].values() for t in L.values()]).view(torch.int32))
                for sa, sb in zip(a, b))
    del a, b
    solo_ms, pop_ms = [], []
    for rep in range(reps):
        for name in (("solo", "pop") if rep % 2 == 0 else ("pop", "solo")):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = run_solo() if name == "solo" else run_pop()
            torch.cuda.synchronize()
            (solo_ms if name == "solo" else pop_ms).append((time.perf_counter() - t0) * 1e3)
            del out
    med = lambda x: sorted(x)[len(x) // 2]  # noqa: E731
    return dict(K=K, solo_ms=solo_ms, grouped_ms=pop_ms, solo_median_ms=med(solo_ms), grouped_median_ms=med(pop_ms),
                speedup=med(solo_ms) / med(pop_ms), params_bit_equal=equal,
                grouped_update_peak_bytes_per_learner=pop_peak / K,
                grouped_scratch_bytes_per_learner=ops.ppo_grad_grouped_scratch_bytes(K, mbs) / K,
                optimizer_steps_per_learner=epochs * (T * n // mbs))


def bench_iterations(K, iterations, reps):
    T, n = 32, 8192
    configs = [dict(seed=k, lr=1e-6 * (1 + k), ent_coef=0.001 * (1 + k), save_model=False, total_timesteps=T * n * iterations)
               for k in range(K)]
    tables = [synthetic_deal_table(100_000, seed=k) for k in range(2)]
    eval_table = synthetic_deal_table(100_000, seed=10_000)

    def stamps():
        out = []
        return out, (lambda log: out.append(time.perf_counter()))

    def per_iter(ts):
        return [b - a for a, b in zip(ts, ts[1:])]  # iterations 1 .. N-1: between consecutive logs

    solo_ms, pop_ms, peak = [], [], {"solo": 0, "pop": 0}
    for rep in range(reps):
        for name in (("solo", "pop") if rep % 2 == 0 else ("pop", "solo")):
            torch.cuda.reset_peak_memory_stats()
            if name == "solo":
                total = None
                for k in range(K):
                    ts, fn = stamps()
                    ppo.train(configs[k], brandom.PRNGKey(k), tables=tables, eval_table=eval_table, log_fn=fn)
                    d = per_iter(ts)
                    total = d if total is None else [a + b for a, b in zip(total, d)]
                solo_ms += [1e3 * x for x in total]
            else:
                ts, fn = stamps()
                ppo.train_population(configs, [brandom.PRNGKey(k) for k in range(K)], tables=tables, eval_table=eval_table,
                                     log_fns=[fn] + [None] * (K - 1))
                pop_ms += [1e3 * x for x in per_iter(ts)]
            peak[name] = max(peak[name], torch.cuda.max_memory_allocated())
            torch.cuda.empty_cache()
    med = lambda x: sorted(x)[len(x) // 2]  # noqa: E731
    return dict(K=K, iterations_per_run=iterations, solo_iteration_ms=solo_ms, population_iteration_ms=pop_ms,
                solo_median_ms=med(solo_ms), population_median_ms=med(pop_ms), speedup=med(solo_ms) / med(pop_ms),
                solo_run_peak_bytes=peak["solo"], population_run_peak_bytes_per_learner=peak["pop"] / K)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--ks", type=int, nargs="*", default=[1, 2, 4, 8])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--num-envs", type=int, default=8192)
    ap.add_argument("--num-steps", type=int, default=32)
    ap.add_argument("--minibatch-size", type=int, default=1024)
    ap.add_argument("--update-epochs", type=int, default=10)
    ap.add_argument("--iter-ks", type=int, nargs="*", default=[1, 2, 4])
    ap.add_argument("--iterations", type=int, default=4)
    ap.add_argument("--iter-reps", type=int, default=2)
    ap.add_argument("--out")
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("population_bench needs a CUDA device")
    res = dict(device=_gpu_label(), num_envs=a.num_envs, num_steps=a.num_steps, minibatch_size=a.minibatch_size,
               update_epochs=a.update_epochs, reps=a.reps, results=[], iterations=[])
    for K in a.ks:
        r = bench_k(K, a.num_steps, a.num_envs, a.minibatch_size, a.update_epochs, a.reps)
        print(json.dumps(r), flush=True)
        res["results"].append(r)
        torch.cuda.empty_cache()
    for K in a.iter_ks:
        r = bench_iterations(K, a.iterations, a.iter_reps)
        print(json.dumps(r), flush=True)
        res["iterations"].append(r)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k not in ("results", "iterations")}))


if __name__ == "__main__":
    main()
