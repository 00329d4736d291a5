"""List the stream operations of one call of each PPO / SL update op, as torch.profiler records them.

    python scripts/launch_sequence.py [--root TREE] [--out listing.txt]

For each case (ppo_grad and ppo_grad_grouped at K = 3, both tile-width tune settings, reward scaling on and off, the
illegal-action statistic on and off; sl_grad and sl_eval) one call is captured after a warm-up call.  Its runtime API
calls are listed in the order the host made them, then its kernels (name, grid, block, dynamic shared memory) and memsets
(bytes) in stream order.  A plain launch lists as cudaLaunchKernel, a programmatic dependent launch as cudaLaunchKernelExC.  Run it on two trees
(--root imports brl_b200 from there) and diff the listings: a host-side refactor must leave them equal."""
import argparse
import json
import os
import sys
import tempfile

ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--out")
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from brl_b200 import _lib, ops  # noqa: E402

DEV = "cuda"
B, TOTAL, K = 1024, 4096, 3


def _rollout(g):
    mask = torch.rand((TOTAL, 38), generator=g, device=DEV) < 0.5
    mask[:, 0] = True
    return dict(obs=(torch.rand((TOTAL, 480), generator=g, device=DEV) < 0.04).to(torch.bfloat16), mask=mask.view(torch.uint8),
                action=torch.multinomial(mask.float(), 1, generator=g)[:, 0].to(torch.int32),
                old_log_prob=-torch.rand(TOTAL, generator=g, device=DEV) * 3, old_value=torch.randn(TOTAL, generator=g, device=DEV),
                adv=torch.randn(TOTAL, generator=g, device=DEV), targets=torch.randn(TOTAL, generator=g, device=DEV),
                index=torch.randperm(TOTAL, generator=torch.Generator().manual_seed(0))[:B].to(DEV, torch.int32))


def _net(k):
    torch.manual_seed(k)
    return torch.randn(ops.mlp_num_params(), device=DEV) * 0.02


def cases():
    g = torch.Generator(device=DEV).manual_seed(1)
    rolls = [_rollout(g) for _ in range(K)]
    r = rolls[0]
    blob = ops.mlp_pack_train(_net(0))
    scratch = ops.mlp_train_scratch(B, DEV)
    grads = torch.empty(ops.mlp_num_params(), device=DEV)
    stats = torch.zeros(8, device=DEV)
    acc = ops.ppo_scratch(DEV)
    stride, nb = ops.mlp_param_stride(), int(_lib.load().brl_mlp_train_blob_bytes())
    gblob = torch.empty((K, nb), dtype=torch.uint8, device=DEV)
    for k in range(K):
        ops.mlp_pack_train(_net(k), out=gblob[k])
    gscratch = torch.empty(ops.ppo_grad_grouped_scratch_bytes(K, B), dtype=torch.uint8, device=DEV)
    ggrads = torch.empty((K, stride), device=DEV)
    gstats = torch.zeros((K, 8), device=DEV)
    gacc = torch.zeros((K, _lib.PPO_SCRATCH_BYTES // 8), dtype=torch.float64, device=DEV)
    table = torch.tensor([ops.ppo_trajectory_row(q["obs"], q["index"], q["mask"], q["action"], q["old_log_prob"], q["old_value"],
                                                 q["adv"], q["targets"]) for q in rolls], dtype=torch.int64).to(DEV)
    coefs = torch.tensor([[0.2, 0.01 * (k + 1), 0.5, 0.0] for k in range(K)], device=DEV)
    for tune in (0, 4 | 16):
        for rs in (False, True):
            for stat in (False, True):
                name = f"tune={tune} reward_scaling={int(rs)} illegal_stat={int(stat)}"
                yield f"ppo_grad {name}", lambda: ops.ppo_grad(
                    r["obs"], blob, scratch, r["index"], r["mask"], r["action"], r["old_log_prob"], r["old_value"], r["adv"],
                    r["targets"], grads, stats, acc, clip_eps=0.2, ent_coef=0.01, vf_coef=0.5, reward_scaling=rs,
                    illegal_stat=stat, tune=tune)
                yield f"ppo_grad_grouped K={K} {name}", lambda: ops.ppo_grad_grouped(
                    table, coefs, gblob, gscratch, ggrads, gstats, gacc, batch=B, obs_dtype=torch.bfloat16, reward_scaling=rs,
                    illegal_stat=stat, tune=tune)
    label = r["action"][:B].clone()
    sl_acc = ops.sl_acc(DEV)
    yield "sl_grad", lambda: ops.sl_grad(r["obs"][:B], blob, scratch, r["mask"][:B], label, grads, stats, sl_acc)
    yield "sl_eval", lambda: ops.sl_eval(r["obs"][:B], blob, scratch, r["mask"][:B], label, stats, sl_acc)


def capture(fn):
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    # host calls in host order, then device work in stream order: the two clocks' relative order is not reproducible
    api, dev = [], []
    for e in sorted((e for e in events if e.get("ph") == "X"), key=lambda e: e["ts"]):
        cat, a = e.get("cat"), e.get("args", {})
        if cat == "cuda_runtime" and e["name"] not in ("cudaDeviceSynchronize", "cudaStreamIsCapturing", "cudaGetLastError"):
            api.append(f"  api     {e['name']}")
        elif cat == "kernel":
            dev.append(f"  kernel  {e['name']}  grid {a.get('grid')}  block {a.get('block')}  smem {a.get('shared memory')}")
        elif cat == "gpu_memset":
            dev.append(f"  memset  {a.get('bytes')} bytes")
    return api + dev


def main():
    out = []
    for name, fn in cases():
        out.append(name)
        out += capture(fn)
    text = "\n".join(out) + "\n"
    sys.stdout.write(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
