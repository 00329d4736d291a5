#!/usr/bin/env python
"""bench.py -- bridge-bidding env-steps/sec (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--sweep] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): random-legal-action env stepping, 8192 envs per
GPU, env only (no policy net).  One bench "step" = one pass of the hot path over one
batch = ONE launch of the fused rollout kernel: 32 auto-reset env sub-steps
(`num_steps`, ppo.py:120) over 8192 envs (`num_envs`, ppo.py:119) = 262,144 env-steps,
writing the full [32, 8192, ...] trajectory (observation f32[480], legal mask, rewards,
terminated, current player, action) = 519 MB per step, which is larger than the 126 MB
L2, so every timed step's stores are DRAM traffic (no flush needed).

Prints ONE JSON line (rank 0).  `value` = whole-job env-steps/s with state resident in
HBM; `e2e` = the same metric through the host-buffer C-ABI (`brl_env_rollout_host`):
per step the action randomness comes from pinned host memory and the rewards /
terminated / statistics go back to pinned host memory, copies inside the timed region
(`e2e.full_io` = every Env-surface output copied out per env.step, PCIe-bound);
`roofline` = the rollout kernel against measured
HBM bandwidth; `cpu_baseline` = the C oracle on this box's host cores (bounded sample).
`--impl reference` times the CPU restatement of the reference on the same config (the
real pgx/JAX env cannot be installed in this image -- see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_ENVS = 8192          # per GPU (ppo.py:119)
T_STEPS = 32           # env sub-steps per launch (ppo.py:120)
N_DEALS = 100_000      # hash_size (ppo.py:128)
BYTES_PER_ENV_STEP = 1980  # SURVEY 8d: obs 1920 + mask 38 + rewards 16 + terminated 1 + player 1 + action 4
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
SEED = 20241017


class _StdoutToStderr:
    """NCCL prints its version banner on fd 1 when the communicator is created; the contract is ONE JSON line on
    stdout, so fd 1 points at stderr while torch.distributed / NCCL initialise."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)
        return False


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _traffic(kernel_key):
    """per-launch DRAM bytes of the bench kernel from the committed `ncu --set full` capture (profiles/)"""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as fh:
            doc = json.load(fh)
            e = doc[doc.get("_alias", {}).get(kernel_key, kernel_key)]
        return e["traffic_bytes"], f"profiles/r02_traffic.json ({e['report']}: dram__bytes_read.sum + dram__bytes_write.sum, mean of {e['instances']} launches)"
    except Exception:
        return None, "no ncu capture committed for this kernel"


def cpu_oracle_throughput(n_envs, t_steps, reps, n_threads, table):
    """env-steps/s of the C oracle (all outputs written, same workload shape)."""
    import numpy as np
    from oracle import oracle as orc
    env = orc.OracleEnv(table, n_envs, n_threads=n_threads)
    env.init(orc.make_keys(SEED, n_envs))
    k, n = t_steps, n_envs
    out = dict(obs=np.zeros((k, n, 480), np.float32), mask=np.zeros((k, n, 38), np.uint8),
               rew=np.zeros((k, n, 4), np.float32), term=np.zeros((k, n), np.uint8), cur=np.zeros((k, n), np.int8),
               act=np.zeros((k, n), np.int32))
    import ctypes as C

    def run(step0):
        return env.L.orc_rollout_random(
            orc._p(env.buf), C.byref(env.params), C.c_int64(n), C.c_int64(0), C.c_uint64(SEED), C.c_uint32(step0),
            C.c_int32(k), orc._p(out["obs"]), orc._p(out["mask"]), orc._p(out["rew"]), orc._p(out["term"]),
            orc._p(out["cur"]), orc._p(out["act"]), C.c_int(n_threads))

    run(0)  # warm-up (page faults of the output buffers)
    times = []
    for r in range(reps):
        t0 = time.perf_counter()
        run((r + 1) * k)
        times.append(time.perf_counter() - t0)
    return n * k * len(times) / sum(times), times


def _oracle_build():
    from oracle import oracle as orc
    return "gcc -O3 -march=" + ("x86-64-v3 (AVX2/BMI2/FMA)" if orc.so_path().endswith("_v3.so") else "x86-64-v2") + ", pthreads"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from brl_b200.deals import synthetic_deal_table
    cores = os.cpu_count() or 1
    table = synthetic_deal_table(N_DEALS, seed=0)
    for _ in range(max(0, args.warmup - 1)):
        cpu_oracle_throughput(N_ENVS, T_STEPS, 1, cores, table)
    value, times = cpu_oracle_throughput(N_ENVS, T_STEPS, args.steps, cores, table)
    ms = 1e3 * sum(times) / len(times)
    sample = f"{args.steps} x ({N_ENVS} envs x {T_STEPS} auto-reset random-legal steps), all outputs written"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8/int32 state, f32 0/1 observation", "data": "synthetic",
        "config": _config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "build": _oracle_build(),
                         "note": "C restatement of pgx 1.4.0 bridge_bidding semantics (oracle/brl_oracle.c), not pgx: "
                                 "jax/pgx are not installable in this image.  It rebuilds the observation from the call "
                                 "list every step, as the reference does; a reported baseline, not a tuned CPU port"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def _config(n_gpus):
    return {"workload": "configs[1]: random-legal-action bridge_bidding env step, 8192 envs per GPU, env only",
            "n_envs_per_gpu": N_ENVS, "env_steps_per_bench_step": N_ENVS * T_STEPS, "sub_steps_per_launch": T_STEPS,
            "n_deals": N_DEALS, "auto_reset": True, "obs_dtype": "f32", "sharding": f"env index x{n_gpus}, no collective in step",
            "l2": "trajectory written per step = 519 MB > 126 MB L2 (no flush needed)"}


DUMP_ENVS = 512  # envs of the [32, 8192, ...] trajectory written by --dump-outputs: 34 MB in all


def dump_outputs(out_dir, np, traj, actions, stats):
    """What a caller of the timed path receives after its last step, as float32 / float64 .npy files, so that two builds
    can be compared output for output.  The full observation trajectory is 503 MB, so every per-env array is cut to the
    same fixed, seeded sample of DUMP_ENVS env columns (sorted); the statistics are the i64[4] sums over the timed steps."""
    os.makedirs(out_dir, exist_ok=True)
    cols = np.sort(np.random.default_rng(SEED).choice(traj.terminated.shape[1], DUMP_ENVS, replace=False))
    arrays = {"observation": traj.observation, "legal_action_mask": traj.legal_action_mask, "rewards": traj.rewards,
              "terminated": traj.terminated, "current_player": traj.current_player, "action": actions}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy()[:, cols].astype(np.float32))
    np.save(os.path.join(out_dir, "episode_stats.npy"), stats.cpu().numpy().astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--sweep", action="store_true", help="also time 65,536 and 1,048,576 envs and single-step launches")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-policy", action="store_true", help="skip the configs[2] policy-rollout leg")
    ap.add_argument("--no-update", action="store_true", help="skip the PPO-update leg (SURVEY 8f-1)")
    ap.add_argument("--no-matches", action="store_true", help="skip the configs[0] / [3] / [4] duplicate-match legs")
    ap.add_argument("--league", action="store_true", help="run the configs[4] 1M-env league leg below 8 GPUs too")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0's trajectory, sampled; the statistics) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    from brl_b200 import _lib, ops
    from brl_b200.deals import synthetic_deal_table

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        with _StdoutToStderr():
            import datetime
            # a rank that dies or skips a collective must fail the run within minutes, not hold 8 GPUs for NCCL's default 10
            dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=150))
            dist.barrier()  # creates the communicator (and prints NCCL's banner) now
    _lib.load()  # fail loudly if the CUDA library is missing

    table_np = synthetic_deal_table(N_DEALS, seed=0)
    table = torch.as_tensor(table_np, device=dev)
    n, k = N_ENVS, T_STEPS
    offset = rank * n  # global env index: results do not depend on the GPU count
    state = ops.new_state(n, dev)
    out0 = ops.EnvOutputs(n, dev)
    ops.init(ops.make_keys(SEED, n, dev, env_offset=offset), table, state, out0)
    traj = ops.EnvOutputs(n, dev, rows=k)
    actions = torch.empty((k, n), dtype=torch.int32, device=dev)
    stats = torch.zeros(4, dtype=torch.int64, device=dev)

    def one_step(i):
        ops.rollout_random(state, table, k, traj, seed=SEED, step0=i * k, env_offset=offset, action_out=actions,
                           stats=stats)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_stats():
        # the single collective of the path: episode statistics summed over ranks (SURVEY 8e).  The rollout kernel
        # accumulates them as integers (exact), so the NCCL all-reduce runs on the kernel's own i64[4] buffer in place:
        # no torch kernel between the last launch and the collective.
        if world > 1:
            dist.all_reduce(stats)
        return stats

    for i in range(args.warmup):
        one_step(i)
    reduce_stats()  # warm the NCCL kernel outside the timed region
    barrier()
    stats.zero_()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # Two events bracket the K launches (a third closes the region after the statistics all-reduce).  An event record after
    # every launch, as earlier revisions had, costs 2.6 us per step on this stream (scripts/exp_bench_overheads.py).
    begin, last, end = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    barrier()
    if world > 1:
        # line the ranks' STREAMS up as well: the host barrier above leaves tens of microseconds of skew between the ranks'
        # first launches, which the closing all-reduce would turn into waiting time on the early ranks.  After this
        # (untimed) collective every rank's timed region starts within NCCL's own completion skew.
        dist.all_reduce(torch.zeros(1, device=dev))
    begin.record()
    for i in range(args.steps):
        one_step(args.warmup + i)
    last.record()
    sums = reduce_stats()
    end.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    total_ms = begin.elapsed_time(end)
    kernel_ms = [begin.elapsed_time(last) / args.steps] * args.steps  # back-to-back launches of the one kernel of a step
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    env_steps = n * k * args.steps * world
    value = env_steps / (total_ms * 1e-3)
    avg_kernel_ms = sum(kernel_ms) / len(kernel_ms)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, np, traj, actions, sums)
    peak, peak_src = _peaks()
    achieved = BYTES_PER_ENV_STEP * n * k / (avg_kernel_ms * 1e-3) / 1e9
    traffic, traffic_src = _traffic("bench_rollout")

    # ---- e2e: host-buffer C-ABI, copies inside the timed region (rank-local, summed over ranks) ----
    e2e = run_e2e(torch, np, _lib, table_np, n, offset, dev, world, dist, steps=max(20, min(200, args.steps * 4)),
                  warmup=args.warmup)

    extra = {}

    def leg(name, fn):
        """a secondary leg must never take the headline line down with it: its failure is recorded, not raised"""
        try:
            extra[name] = fn()
        except Exception as exc:  # noqa: BLE001
            import traceback
            traceback.print_exc(file=sys.stderr)
            extra[name] = {"error": f"{type(exc).__name__}: {exc}"}

    # ---- the north-star multi-GPU configs (all ranks take part; one all-reduce each) ----------------------------------
    if not args.no_matches:
        leg("dup_selfplay_65536", lambda: run_dup_selfplay(torch, dist, dev, rank, world, table_np))
        if world >= 8 or args.league:
            leg("league_1M", lambda: run_league(torch, dist, dev, rank, world, table_np))
        if rank == 0:
            leg("c1_eval_match", lambda: run_c1(torch, dev))
    if args.sweep and rank == 0:
        leg("sweep", lambda: run_sweep(torch, ops, table, dev, peak))
    if rank == 0 and not args.no_policy:
        leg("policy_rollout", lambda: run_policy_rollout(torch, table_np, dev))
    if rank == 0 and not args.no_update:
        leg("ppo_update", lambda: run_ppo_update(torch, dev))

    cpu = None
    if rank == 0 and not args.no_cpu:
        try:
            cores = os.cpu_count() or 1
            reps = 100  # ~1.2 s wall x all cores = 10-30 s of CPU work
            v, times = cpu_oracle_throughput(n, k, reps, cores, table_np)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{reps} x ({n} envs x {k} auto-reset random-legal steps), all outputs written, {cores} threads, "
                             f"{sum(times):.2f} s wall",
                   "build": _oracle_build(),
                   "note": "C restatement of pgx semantics (oracle/brl_oracle.c); pgx/JAX not installable here.  It rebuilds the "
                           "observation from the call list every step, as the reference does: a reported baseline, not a tuned "
                           "CPU port -- the roofline fraction, not this ratio, says how good the kernel is"}
        except Exception as exc:  # noqa: BLE001
            cpu = {"error": f"{type(exc).__name__}: {exc}"}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/int32 state, f32 0/1 observation", "data": "synthetic", "config": _config(world),
            "e2e": e2e, "gpu_launches": args.steps,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel": "brl::k_rollout_ws<f32> (296 blocks = 2 per SM, 27-28 envs each: 1 env warp + 4 writer warps)", "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": BYTES_PER_ENV_STEP * n * k, "avg_launch_ms": avg_kernel_ms,
                         "note": "write-only stream; at 8192 envs per GPU the limiter is the SM-side store path, not DRAM "
                                 "(profiles/r02_n_rollout_decomposition.txt); the same kernel reaches 0.92 at 65,536 envs"},
            "cpu_baseline": cpu, "clocks": clocks,
            "episode_stats": {"finished_auctions": float(sums[0]), "sum_reward_player0": float(sums[1]),
                              "env_steps": float(sums[2]), "collective": "1 NCCL all-reduce of i64[4], in place on the kernel's statistics buffer" if world > 1 else "none (1 rank)"},
        }
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_e2e(torch, np, _lib, table_np, n, offset, dev, world, dist, steps, warmup):
    """Public host-buffer C-ABI, copies inside the timed region.

    `e2e` (headline): one `brl_env_rollout_host_compact_async` call per bench step = the same 32 x 8192 env-steps as
    `value`, three calls in flight.  HOST in: the randomness of the action choice from pinned memory (the `action` input
    of the algorithmic byte count; the host owns the PRNG stream the way the reference's host owns the jax key) as
    u32[32, 8192] (4 B per env-step; the k-th legal action is (u * #legal) >> 32).  HOST out: the step's result as
    i16[32, 8192] = 2 * rewards[player 0] + terminated -- lossless for rewards f32[.., 4] + terminated u8, which is what
    roll_out's consumer reads (src/roll_out.py:86-94) -- + the statistics vector.  The observation / mask / f32 reward
    trajectories stay in HBM for the device-resident consumer, exactly as `traj_batch` does in the reference
    (src/roll_out.py:105-108).  Sub-entries: `u16_uniforms` (2 B/env-step in: half the H2D bytes, but its kernel is 2 %
    slower and at 1-8 GPUs of this pool it never wins -- profiles/r02_*bench*), `f32_payload` (round 1's
    payload: u32 in, rewards f32[4] + terminated u8 out = 17 B/env-step), `sync_per_call` (f32 payload, blocking).
    `full_io`: the other extreme -- one env.step per call with EVERY Env-surface output copied to the host (PCIe-bound
    by construction: 536 B per env-step in pgx's bool observation dtype)."""
    import ctypes as C
    L = _lib.load()
    tbl = np.ascontiguousarray(table_np)
    k = T_STEPS
    rng = np.random.default_rng(SEED + offset)
    n_pool = min(steps + warmup, 16)  # pre-generated host randomness ("the dataset"), cycled
    pool32 = torch.from_numpy(rng.integers(0, 2 ** 32, size=(n_pool, k, n), dtype=np.uint32).view(np.int32)).pin_memory()
    pool16 = torch.from_numpy((pool32.numpy().view(np.uint32) >> 16).astype(np.uint16).view(np.int16)).pin_memory()
    vp = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    depth = max(1, min(4, int(os.environ.get("BRL_E2E_DEPTH", "3"))))  # BRL_ENV_PIPELINE_DEPTH = 4 staging slots

    def timed(fn_loop):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn_loop()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def leg(kind):
        """kind: 'compact16' | 'compact32' | 'f32'.  Returns (seconds for `steps` pipelined calls, finished auctions the
        host read, seconds for `steps` blocking calls or None)."""
        flags = _lib.F_AUTORESET | (_lib.F_UNIFORM_U16 if kind == "compact16" else 0)
        h = L.brl_env_create(n, offset, tbl.ctypes.data, tbl.shape[0], SEED, flags)
        if not h:
            raise RuntimeError("brl_env_create failed: " + L.brl_last_error().decode())
        rc = L.brl_env_init_host(h, None, None, None, None, None)
        assert rc == 0, L.brl_last_error()
        pool = pool16 if kind == "compact16" else pool32
        stats = [torch.zeros(4, dtype=torch.int64).pin_memory() for _ in range(depth)]
        if kind == "f32":
            rew = [torch.zeros((k, n, 4), dtype=torch.float32).pin_memory() for _ in range(depth)]
            term = [torch.zeros((k, n), dtype=torch.uint8).pin_memory() for _ in range(depth)]
            submit = lambda i, j: L.brl_env_rollout_host_async(h, k, vp(pool[i % n_pool]), vp(rew[j]), vp(term[j]), vp(stats[j]))  # noqa: E731
        else:
            res = [torch.zeros((k, n), dtype=torch.int16).pin_memory() for _ in range(depth)]
            submit = lambda i, j: L.brl_env_rollout_host_compact_async(h, k, vp(pool[i % n_pool]), vp(res[j]), vp(stats[j]))  # noqa: E731
        seen = [0]

        def pipelined(count, base):
            inflight = []
            for i in range(count):
                j = i % depth
                if len(inflight) == depth:  # slot j's host buffers are about to be reused: consume their result first
                    t0_, j0 = inflight.pop(0)
                    if L.brl_env_wait(h, t0_) != 0:
                        raise RuntimeError(L.brl_last_error().decode())
                    seen[0] += int(stats[j0][0])   # the host consumes an older step's result while newer ones run
                t = submit(base + i, j)
                if t <= 0:
                    raise RuntimeError(L.brl_last_error().decode())
                inflight.append((t, j))
            for t0_, j0 in inflight:
                if L.brl_env_wait(h, t0_) != 0:
                    raise RuntimeError(L.brl_last_error().decode())
                seen[0] += int(stats[j0][0])

        pipelined(warmup, 0)
        seen[0] = 0
        dt = timed(lambda: pipelined(steps, warmup))
        finished = seen[0]
        dt_sync = None
        if kind == "f32":  # one blocking call per bench step (results written in place into the pinned buffers)
            def one(i):
                if L.brl_env_rollout_host(h, k, vp(pool[i % n_pool]), vp(rew[0]), vp(term[0]), vp(stats[0])) != 0:
                    raise RuntimeError(L.brl_last_error().decode())
            for i in range(warmup):
                one(i)
            dt_sync = timed(lambda: [one(warmup + i) for i in range(steps)])
        L.brl_env_destroy(h)
        return dt, finished, dt_sync

    dt32, finished, _ = leg("compact32")
    dt16, _, _ = leg("compact16")
    dtf, _, dt_sync = leg("f32")
    tot = n * k * steps * world
    res = {"value": tot / dt32, "unit": UNIT, "h2d_bytes_per_step": n * k * 4, "d2h_bytes_per_step": n * k * 2 + 32,
           "steps": steps, "ms_per_step": 1e3 * dt32 / steps,
           "api": "brl_env_rollout_host_compact_async + brl_env_wait (C ABI, host buffers), three calls in flight: per bench "
                  "step H2D u32[32,8192] action randomness from pinned memory, one fused rollout launch writing the full "
                  "trajectory (incl. f32 rewards / u8 terminated) to HBM, D2H result i16[32,8192] = 2*rewards[player 0] + "
                  "terminated (lossless: rewards are s*[+,+,-,-]) + stats into pinned memory, read by the host while the next "
                  "steps compute; obs/mask trajectories stay in HBM for the device-resident learner (as traj_batch does "
                  "in the reference)",
           "timed_with": "host wall clock around the whole loop, max over ranks", "finished_auctions_read_on_host": finished,
           "u16_uniforms": {"value": tot / dt16, "ms_per_step": 1e3 * dt16 / steps, "h2d_bytes_per_step": n * k * 2,
                            "d2h_bytes_per_step": n * k * 2 + 32},
           "f32_payload": {"value": tot / dtf, "ms_per_step": 1e3 * dtf / steps, "h2d_bytes_per_step": n * k * 4,
                           "d2h_bytes_per_step": n * k * 17 + 32,
                           "api": "brl_env_rollout_host_async: u32 uniforms in, rewards f32[32,8192,4] + terminated u8 out "
                                  "(round 1's e2e payload)"},
           "sync_per_call": {"value": tot / dt_sync, "ms_per_step": 1e3 * dt_sync / steps,
                             "api": "brl_env_rollout_host: f32 payload, one blocking call per step (results written in place "
                                    "into the pinned buffers by the kernel, no overlap between steps)"}}

    # ---- full I/O: every Env-surface output to the host, one env.step per call -------------------
    h = L.brl_env_create(n, offset, tbl.ctypes.data, tbl.shape[0], SEED, _lib.F_AUTORESET | _lib.F_OBS_U8)
    pin = dict(act=torch.zeros(n, dtype=torch.int32).pin_memory(), obs=torch.zeros((n, 480), dtype=torch.uint8).pin_memory(),
               mask=torch.zeros((n, 38), dtype=torch.uint8).pin_memory(), rew=torch.zeros((n, 4), dtype=torch.float32).pin_memory(),
               term=torch.zeros(n, dtype=torch.uint8).pin_memory(), cur=torch.zeros(n, dtype=torch.int8).pin_memory())
    p = {kk: vp(v) for kk, v in pin.items()}
    rc = L.brl_env_init_host(h, p["obs"], p["mask"], p["rew"], p["term"], p["cur"])
    assert rc == 0, L.brl_last_error()
    mask_np, act_np = pin["mask"].numpy(), pin["act"].numpy()
    passes = rng.random((64, n)) < 0.6

    def host_policy(i):
        # host-side legal choice from the mask that came back over PCIe: pass, or the cheapest bid
        first_bid = mask_np[:, 3:].argmax(axis=1) + 3
        has_bid = mask_np[np.arange(n), first_bid] != 0
        act_np[:] = np.where(passes[i % 64] | ~has_bid, 0, first_bid)

    fsteps = 60
    for i in range(3):
        host_policy(i)
        L.brl_env_step_host(h, p["act"], p["obs"], p["mask"], p["rew"], p["term"], p["cur"])
    t_pol = t_call = 0.0
    for i in range(fsteps):
        a = time.perf_counter()
        host_policy(i)
        b = time.perf_counter()
        rc = L.brl_env_step_host(h, p["act"], p["obs"], p["mask"], p["rew"], p["term"], p["cur"])
        t_call += time.perf_counter() - b
        t_pol += b - a
        if rc != 0:
            raise RuntimeError(L.brl_last_error().decode())
    L.brl_env_destroy(h)
    res["full_io"] = {"value": n * fsteps / (t_pol + t_call), "value_excluding_host_policy": n * fsteps / t_call, "unit": UNIT,
                      "h2d_bytes_per_step": n * 4, "d2h_bytes_per_step": n * (480 + 38 + 16 + 1 + 1),
                      "ms_per_call": 1e3 * t_call / fsteps, "ms_host_policy": 1e3 * t_pol / fsteps, "rank": "0 only" if world > 1 else "0",
                      "api": "brl_env_step_host: 1 env.step over 8192 envs per call, actions from the host, observation (pgx bool/u8), "
                             "mask, rewards, terminated, current_player all copied to pinned host memory"}
    return res


def _weights(name):
    """bundled model pickle of the reference (15 MB each, not in the repository) if copied to tests/golden/_weights"""
    path = os.path.join(ROOT, "tests", "golden", "_weights", name)
    return path if os.path.exists(path) else None


def _timed_match(torch, dist, dev, world, fn, reps):
    """CUDA-event time of `fn()` (which ends in its own all-reduce), max over ranks; best of `reps` after one warm-up"""
    fn()
    best, res = None, None
    for _ in range(reps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        best = float(t) if best is None else min(best, float(t))
    return best, res


def run_dup_selfplay(torch, dist, dev, rank, world, table_np, n_total=65536):
    """BASELINE.json configs[3]: duplicate self-play match (src/evaluation.py:69-204), 65,536 envs in total sharded by
    GLOBAL env index over the ranks (strong scaling: the total is fixed), one all-reduce of the f64[8] IMP statistics.
    Keys use global indices, so the statistics are identical for every rank count."""
    from brl_b200 import BridgeBidding, dist as bdist, random as brandom
    from brl_b200.evaluation import make_simple_duplicate_evaluate
    from brl_b200.models import init_params, load_params
    lo, hi = bdist.shard_range(n_total, rank, world)
    env = BridgeBidding(table=table_np, device=dev)
    w1, w2 = _weights("model-pretrained-rl.pkl"), _weights("model-pretrained-rl-with-fsp.pkl")
    if w1 and w2:
        p1, p2, who = load_params(w1, dev), load_params(w2, dev), "model-pretrained-rl.pkl vs model-pretrained-rl-with-fsp.pkl (bundled weights)"
    else:
        p1, p2, who = init_params(1, dev), init_params(2, dev), "random-init nets (weight fixtures missing)"
    evaluate = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", hi - lo, env_offset=lo)
    ms, res = _timed_match(torch, dist, dev, world, lambda: evaluate(p1, p2, brandom.PRNGKey(1)), reps=2)
    (mean, se, win), _, _, _ = res
    fwd = torch.tensor([float(evaluate.rows_forwarded)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(fwd)
    return {"workload": "configs[3]: duplicate self-play, 65,536 envs total, DeepMind MLP per team, argmax play; " + who,
            "n_envs_total": n_total, "n_gpus": world, "scaling": "strong", "ms_per_match": ms,
            "boards_per_sec": 2 * n_total / (ms * 1e-3), "env_steps_per_sec": float(fwd) / (ms * 1e-3),
            "net_rows_forwarded": float(fwd), "imp_mean": mean, "imp_se": se, "win_rate": win,
            "collective": "1 NCCL all-reduce of f64[8] per match" if world > 1 else "none (1 rank)",
            "note": "env_steps = live (env, call) pairs = rows sent through a net: each net runs only on the live envs its "
                    "team decides (brl_team_rows + brl_policy_act_rows)"}


def run_league(torch, dist, dev, rank, world, table_np, n_total=1 << 20):
    """BASELINE.json configs[4]: FSP/PFSP league probe (ppo.py:399-440): the learner against the pool of the 5 bundled
    models, 1,048,576 envs in total, block m of the global env range plays pool model m, every block sharded over the
    ranks; one all-reduce of f64[5, 8]."""
    from brl_b200 import BridgeBidding, random as brandom
    from brl_b200.evaluation import make_league_evaluate
    from brl_b200.models import init_params, load_params
    names = ("model-sl.pkl", "model-from-scratch-rl.pkl", "model-pretrained-rl.pkl", "model-pretrained-rl-with-fsp.pkl",
             "model-pretrained-rl-with-pfsp.pkl")
    paths = [_weights(n) for n in names]
    env = BridgeBidding(table=table_np, device=dev)
    if all(paths):
        pool, actor, who = [load_params(p, dev) for p in paths], load_params(paths[2], dev), "bundled weights: learner = model-pretrained-rl"
    else:
        pool, actor, who = [init_params(100 + m, dev) for m in range(5)], init_params(1, dev), "random-init nets (weight fixtures missing)"
    league = make_league_evaluate(env, "relu", "DeepMind", n_total, len(pool))
    ms, res = _timed_match(torch, dist, dev, world, lambda: league(actor, pool, brandom.PRNGKey(1)), reps=1)
    return {"workload": "configs[4]: league probe, learner vs the pool of 5 models, 1,048,576 envs total; " + who,
            "n_envs_total": n_total, "n_gpus": world, "scaling": "strong", "ms_per_league": ms,
            "boards_per_sec": 2 * n_total / (ms * 1e-3), "pool": list(names),
            "imp_mean": [r[0] for r in res], "imp_se": [r[1] for r in res], "win_rate": [r[2] for r in res],
            "collective": "1 NCCL all-reduce of f64[5,8]" if world > 1 else "none (1 rank)"}


def run_c1(torch, dev):
    """BASELINE.json configs[0]: eval.py duplicate match model-pretrained-rl.pkl vs model-sl.pkl, num_eval_envs=100, on the
    1000 real boards (eval.py:43-65).  IMP mean +- SE must equal the golden values the oracle + the reference's own scorer
    produced (tests/golden/make_c1_golden.py); the oracle is not touched here."""
    import numpy as np
    from brl_b200 import BridgeBidding, random as brandom
    from brl_b200.evaluation import make_simple_duplicate_evaluate
    from brl_b200.models import load_params
    w1, w2 = _weights("model-pretrained-rl.pkl"), _weights("model-sl.pkl")
    if not (w1 and w2):
        return {"unavailable": "weight fixtures missing (tests/golden/_weights)"}
    boards = np.load(os.path.join(ROOT, "tests", "golden", "boards_wb5_1000.npz"))["table"]
    gold = np.load(os.path.join(ROOT, "tests", "golden", "c1_eval_match.npz"))
    env = BridgeBidding(table=boards, device=dev)
    p1, p2 = load_params(w1, dev), load_params(w2, dev)
    from brl_b200 import dist as bdist
    evaluate = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", 100)

    def match():  # rank 0 ONLY runs this leg: keep the statistics local (no collective the other ranks never join)
        sums = torch.zeros(8, dtype=torch.float64, device=dev)
        _, _, _, cum = evaluate(p1, p2, brandom.PRNGKey(0), local_sums=sums)
        return bdist.stats_from_sums(sums.cpu()), cum

    ms, res = _timed_match(torch, None, dev, 1, match, reps=3)
    (mean, se, win), cum = res
    return {"workload": "configs[0]: eval.py model-pretrained-rl.pkl vs model-sl.pkl, num_eval_envs=100, 1000 real boards",
            "ms_per_match": ms, "imp_mean": mean, "imp_se": se, "win_rate": win,
            "golden_imp_mean": float(gold["stats"][0]), "golden_imp_se": float(gold["stats"][1]),
            "equals_golden": bool((cum.cpu().numpy() == gold["imps"]).all())}


def run_policy_rollout(torch, table_np, dev):
    """BASELINE.json configs[2]: ppo.py rollout, num_envs=8192, num_steps=32, DeepMind 4x1024 ReLU policy
    (random init) for actor and opponent, competitive quad step, + GAE.  Secondary to the headline metric:
    reported so the tensor-core policy forward has a measured number beside the env kernels."""
    from brl_b200 import BridgeBidding
    from brl_b200 import random as brandom
    from brl_b200.gae import make_calc_gae
    from brl_b200.models import init_params, make_forward_pass
    from brl_b200.roll_out import make_roll_out
    n, T = N_ENVS, T_STEPS
    env = BridgeBidding(table=table_np, device=dev)
    config = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode="competitive",
                  num_steps=T, reward_scale=7600.0, gamma=1.0, gae_lambda=0.95)
    out = {"workload": "configs[2]: ppo.py rollout num_envs=8192 num_steps=32 + GAE, DeepMind MLP random-init; "
                       "1 rollout = 32 x 4 env sub-steps x 8192 envs and 129 policy forwards"}
    flops = 7354368.0 * n
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            tpeak = float(json.load(fh)["bf16_tflops"])
    except Exception:
        tpeak = 1590.0
    from scripts.torch_baseline import TorchForwardPass  # cuBLAS comparison leg only; not a product back end
    for prec in ("tc", "tc-bf16", "fp32"):
        fp = TorchForwardPass("relu", "fp32") if prec == "fp32" else make_forward_pass("relu", "DeepMind", precision=prec)
        params, opp = init_params(1, dev), init_params(2, dev)
        state = env.init(env.make_keys(SEED, n))
        runner = (params, None, state, state.observation, torch.zeros((), dtype=torch.int64, device=dev), brandom.PRNGKey(3))
        roll_out, calc_gae = make_roll_out(config, env, fp, fp), make_calc_gae(config, fp)
        reps = 5 if prec != "fp32" else 1
        for _ in range(2 if prec != "fp32" else 1):  # warm-up (lazy allocations, parameter packing, clocks)
            runner, traj = roll_out(runner, opp)
            calc_gae(runner, traj)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = []
        for _ in range(reps):  # one rollout + GAE per timed interval; the median is reported
            e0.record()
            runner, traj = roll_out(runner, opp)
            calc_gae(runner, traj)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        ms = statistics.median(times)
        x = traj.obs[0]
        for _ in range(3):
            fp.apply(params, x)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(20):
            fp.apply(params, x)
        e1.record()
        torch.cuda.synchronize()
        fms = e0.elapsed_time(e1) / 20
        mma_factor = {"tc": (2 * 480 + 3 * (3 * 1024 + 39)) / (480 + 3 * 1024 + 39.0), "tc-bf16": 1.0}.get(prec)
        out[prec] = {"ms_per_rollout_plus_gae": ms, "ms_min_max": [min(times), max(times)], "env_steps_per_sec": n * T * 4 / (ms * 1e-3),
                     "agent_steps_per_sec": n * T / (ms * 1e-3), "forward_ms_8192": fms,
                     "forward_model_TFLOPs": flops / (fms * 1e-3) / 1e12}
        if mma_factor:
            out[prec]["forward_tensor_roofline"] = {
                "bound": "tensor", "achieved": flops * mma_factor / (fms * 1e-3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                "frac": flops * mma_factor / (fms * 1e-3) / 1e12 / tpeak,
                "note": "achieved = bf16 MMA FLOPs actually issued (x%.2f of the model's FLOPs in this mode) / CUDA-event time of the "
                        "whole forward (obs->bf16 cast + 5 layer launches); peak = measured cuBLAS bf16 burst" % mma_factor}
    return out


def run_ppo_update(torch, dev):
    """SURVEY 8f-1: the update half of a ppo.py iteration on the configs[2] rollout shape (8192 envs x 32 steps,
    minibatch 1024 => 256 optimizer steps per epoch): minibatch take + forward + loss + backward + clip/Adam per
    step, through `make_update_step` (the call ppo.py makes), one epoch per timed call.  "tc" = all hand-written
    kernels (brl_ppo_grad on tcgen05); "fp32" = the same loss / Adam kernels around cuBLAS fp32 GEMMs via autograd."""
    from brl_b200 import random as brandom
    from brl_b200.models import init_params, make_forward_pass
    from brl_b200.optim import AdamWithClip
    from brl_b200.roll_out import Transition
    from brl_b200.update import make_update_step
    n, T, mbs = N_ENVS, T_STEPS, 1024
    nmb = n * T // mbs
    config = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, clip_eps=0.2, ent_coef=0.01, vf_coef=0.5,
                  illegal_action_l2norm_coef=0.0, value_clipping=True, reward_scaling=False, num_minibatches=nmb,
                  minibatch_size=mbs, update_epochs=1, num_steps=T, num_envs=n)
    g = torch.Generator(device=dev).manual_seed(11)
    obs = (torch.rand((T, n, 480), generator=g, device=dev) < 0.04).to(torch.bfloat16)
    mask = torch.rand((T, n, 38), generator=g, device=dev) < 0.5
    mask[..., 0] = True
    traj = Transition(done=torch.zeros((T, n), dtype=torch.bool, device=dev),
                      action=torch.zeros((T, n), dtype=torch.int32, device=dev),
                      value=torch.randn((T, n), generator=g, device=dev) * 0.3, reward=torch.zeros((T, n), device=dev),
                      log_prob=-torch.rand((T, n), generator=g, device=dev) * 3, obs=obs, legal_action_mask=mask)
    adv = torch.randn((T, n), generator=g, device=dev)
    tgt = torch.randn((T, n), generator=g, device=dev) * 0.3
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            tpeak = float(json.load(fh)["bf16_tflops"])
    except Exception:
        tpeak = 1590.0
    model_flop = 3 * 7354368.0 * mbs  # forward + input gradients + weight gradients, per optimizer step
    # bf16 MMA FLOPs the split mode issues per sample: 3 products per term, 2 where the 0/1 observation is an operand
    H, hp = 1024, 64
    mma_flop = 2.0 * mbs * ((480 * H * 2 + 3 * H * H * 3 + H * hp * 3) + (hp * H * 3 + 3 * H * H * 3) + (H * hp * 3 + 3 * H * H * 3 + 480 * H * 2))
    out = {"workload": f"ppo.py update on the configs[2] rollout: {T} x {n} samples, minibatch {mbs}, 1 epoch = {nmb} optimizer steps "
                       "(take + forward + loss + backward + clip_by_global_norm + Adam each); synthetic trajectory, random-init net"}
    from scripts.torch_baseline import TorchForwardPass, make_update_step_autograd  # comparison leg only
    for prec, reps in (("tc", 3), ("fp32", 1)):
        params = init_params(1, dev)
        opt = AdamWithClip(1e-4, eps=1e-5, max_grad_norm=0.5)
        update_step = (make_update_step(config, make_forward_pass("relu", "DeepMind"), opt) if prec == "tc"
                       else make_update_step_autograd(config, TorchForwardPass("relu", "fp32"), opt))
        runner = (params, opt.init(params), None, None, 0, brandom.PRNGKey(5))
        runner, info0 = update_step(runner, traj, adv, tgt)  # warm-up epoch
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            runner, info = update_step(runner, traj, adv, tgt)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps / nmb
        out[prec] = {"ms_per_optimizer_step": ms, "ms_per_epoch": ms * nmb, "samples_per_sec": mbs / (ms * 1e-3),
                     "model_TFLOPs": model_flop / (ms * 1e-3) / 1e12,
                     "first_total_loss": float(info0[0][0, 0])}  # same parameters and minibatch in both back ends
        if prec == "tc":
            out[prec]["tensor_roofline"] = {
                "bound": "tensor", "achieved": mma_flop / (ms * 1e-3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                "frac": mma_flop / (ms * 1e-3) / 1e12 / tpeak,
                "note": "achieved = bf16 MMA FLOPs issued by the 14 split GEMMs of one step / CUDA-event time of the WHOLE optimizer step "
                        "(incl. take, loss, bias sums, Adam, re-pack); a 1024-row minibatch gives each GEMM 64 full-rate 128x128 tiles "
                        "for 148 SMs and every layer is a dependency step, so the launch-level tensor-pipe activity is 19-30 % "
                        "(profiles/r01_m_ppo_update_*, DESIGN.md section 3)"}
    out["speedup_tc_over_library_fp32"] = out["fp32"]["ms_per_optimizer_step"] / out["tc"]["ms_per_optimizer_step"]
    return out


def run_sweep(torch, ops, table, dev, peak):
    """Larger env counts (footprint >> L2 per step) and the one-launch-per-env.step path."""
    from brl_b200 import _lib
    res = []
    n, k = N_ENVS, T_STEPS
    state, out0 = ops.new_state(n, dev), ops.EnvOutputs(n, dev)
    ops.init(ops.make_keys(SEED, n, dev), table, state, out0)
    traj = ops.EnvOutputs(n, dev, rows=k)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, kw in (("ws7", {"writers": 7}), ("ws5", {"writers": 5}), ("ws3", {"writers": 3}), ("ws1", {"writers": 1}),
                     ("tile8", {"classic_rollout": True, "epw": 8}), ("tile16", {"classic_rollout": True, "epw": 16}),
                     ("tile32", {"classic_rollout": True, "epw": 32})):
        tune = _lib.tune(**kw)
        for i in range(3):
            ops.rollout_random(state, table, k, traj, seed=SEED, step0=i * k, tune=tune)
        torch.cuda.synchronize()
        e0.record()
        for i in range(10):
            ops.rollout_random(state, table, k, traj, seed=SEED, step0=(3 + i) * k, tune=tune)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        gbs = BYTES_PER_ENV_STEP * n * k / (ms * 1e-3) / 1e9
        res.append({"kernel": "rollout:" + name, "n_envs": n, "sub_steps": k, "ms": round(ms, 4), "GBps": round(gbs, 1), "frac": round(gbs / peak, 4)})
    del state, out0, traj
    for n, k in ((65536, 8), (1048576, 2)):
        state, out0 = ops.new_state(n, dev), ops.EnvOutputs(n, dev)
        ops.init(ops.make_keys(SEED, n, dev), table, state, out0)
        traj = ops.EnvOutputs(n, dev, rows=k)
        for i in range(3):
            ops.rollout_random(state, table, k, traj, seed=SEED, step0=i * k)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for i in range(reps):
            ops.rollout_random(state, table, k, traj, seed=SEED, step0=(3 + i) * k)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        gbs = BYTES_PER_ENV_STEP * n * k / (ms * 1e-3) / 1e9
        res.append({"kernel": "k_rollout", "n_envs": n, "sub_steps": k, "ms": ms, "env_steps_per_sec": n * k / (ms * 1e-3),
                    "GBps": gbs, "frac": gbs / peak})
        # single env.step per launch (in-kernel random action), outputs to one [n, ...] slot
        out1 = ops.EnvOutputs(n, dev)
        for i in range(3):
            ops.step(state, None, table, state, out1, autoreset=True, random_action=True, seed=SEED, step_index=i)
        torch.cuda.synchronize()
        e0.record()
        for i in range(20):
            ops.step(state, None, table, state, out1, autoreset=True, random_action=True, seed=SEED, step_index=10 + i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 20
        gbs = BYTES_PER_ENV_STEP * n / (ms * 1e-3) / 1e9
        res.append({"kernel": "k_step", "n_envs": n, "ms": ms, "env_steps_per_sec": n / (ms * 1e-3), "GBps": gbs,
                    "frac": gbs / peak})
        del state, out0, traj, out1
        torch.cuda.empty_cache()
    return res


if __name__ == "__main__":
    main()
