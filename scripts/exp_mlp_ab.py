"""A/B of the two MLP forward paths (interleaved, CUDA events): per-layer launches vs the one fused launch, in both
precisions, at batch sizes around the 4096-row switch between them (kPairMinM in brl_b200/csrc/mlp_device.cuh)."""
import os, sys, statistics, torch
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200 import ops
from brl_b200.models import LAYERS, init_params
dev = "cuda:0"
LAYERS_BIT, FUSED_BIT = 1 << 29, 1 << 30  # BRL_F_TUNE_MLP_LAYERS, BRL_F_TUNE_MLP_FUSED (include/brl_b200.h)
sizes = [int(a) for a in sys.argv[1:]] or [1024, 2048, 4096, 8192, 65536]
for n in sizes:
    params = init_params(1, dev)
    for name in LAYERS:
        params[name]["b"] = torch.randn_like(params[name]["b"]) * 0.1
    blob = ops.mlp_pack([params[k]["w"] for k in LAYERS], [params[k]["b"] for k in LAYERS])
    x = (torch.rand((n, 480), device=dev) < 0.05).to(torch.bfloat16)
    scratch = ops.mlp_scratch(n, dev)
    lg, v = torch.empty((n, 38), device=dev), torch.empty(n, device=dev)
    ref = {}
    res = {}
    variants = (("layers x3", {"tune": LAYERS_BIT}), ("fused x3", {"tune": FUSED_BIT}),
                ("layers bf16", {"single_bf16": True, "tune": LAYERS_BIT}), ("fused bf16", {"single_bf16": True, "tune": FUSED_BIT}))
    for rnd in range(5):
        for name, kw in variants:
            lg.fill_(float("nan")); v.fill_(float("nan"))
            for _ in range(3): ops.mlp_forward(x, blob, scratch, lg, v, **kw)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20): ops.mlp_forward(x, blob, scratch, lg, v, **kw)
            e1.record(); torch.cuda.synchronize()
            res.setdefault(name, []).append(e0.elapsed_time(e1) / 20)
            if rnd == 0:
                mode = name.split()[1]
                if mode not in ref:
                    ref[mode] = (lg.clone(), v.clone())
                else:
                    r = ref[mode]
                    print(f"n={n} {name}: bit-equal to layers {mode}: logits {torch.equal(lg, r[0])} value {torch.equal(v, r[1])}"
                          f"  max|d| {float((lg - r[0]).abs().max()):.3g}", flush=True)
    for name, t in res.items():
        m = statistics.median(t)
        print(f"n={n} {name:12s} median {m*1e3:8.1f} us  model TFLOP/s {7354368*n/m/1e9:7.1f}", flush=True)
