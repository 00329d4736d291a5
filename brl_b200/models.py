"""Policy/value net of the rollout and evaluation loops: the "DeepMind" 4x1024 ReLU
actor-critic (src/models.py:23-33); parameters keep haiku's layout
(`actor_critic/linear{,_1..5}` -> {'w' [in,out], 'b'}).

precision (both run the hand-written TMA + tcgen05 forward of csrc/brl_mlp.cu; there is no library back end in the
product -- the cuBLAS cross-check lives in scripts/torch_baseline.py):
  "tc"      3-term bf16 split with fp32 accumulation in tensor memory -- fp32-class results (the reference
            computes in fp32);
  "tc-bf16" a single bf16 product per term.
"""
from __future__ import annotations

import io
import pickle
from typing import Dict

import numpy as np
import torch

from . import ops

LAYERS = ("actor_critic/linear", "actor_critic/linear_1", "actor_critic/linear_2", "actor_critic/linear_3",
          "actor_critic/linear_4", "actor_critic/linear_5")
SIZES = ((480, 1024), (1024, 1024), (1024, 1024), (1024, 1024), (1024, 38), (1024, 1))


class _NoJaxUnpickler(pickle.Unpickler):
    """brl pickles embed `jax._src.array._reconstruct_array`; rebuild plain NumPy instead
    (ppo.py:351-362 writes them, eval.py:56-57 reads them)."""

    def find_class(self, module, name):
        if module.startswith("jax") and name == "_reconstruct_array":
            def rebuild(fun, args, state, aval=None):
                arr = fun(*args)
                arr.__setstate__(state)
                return arr
            return rebuild
        if module.startswith("numpy.core"):
            module = module.replace("numpy.core", "numpy._core", 1)
        return super().find_class(module, name)


def load_params(path: str, device="cuda") -> Dict[str, Dict[str, torch.Tensor]]:
    with open(path, "rb") as fh:
        raw = _NoJaxUnpickler(io.BytesIO(fh.read())).load()
    return {k: {n: torch.as_tensor(np.asarray(a, dtype=np.float32), device=device) for n, a in v.items()}
            for k, v in raw.items()}


def check_params_file(path: str) -> None:
    """ValueError unless the pickle at `path` holds a DeepMind 4x1024 net (the LAYERS, each 'w' / 'b' of the SIZES), read on
    the host only -- so a wrong file is refused before any device work"""
    with open(path, "rb") as fh:
        raw = _NoJaxUnpickler(io.BytesIO(fh.read())).load()
    if not isinstance(raw, dict) or set(raw) != set(LAYERS):
        raise ValueError(f"{path}: not a DeepMind 4x1024 parameter set (layers {sorted(raw) if isinstance(raw, dict) else type(raw)})")
    for name, (fi, fo) in zip(LAYERS, SIZES):
        shapes = {k: tuple(np.shape(raw[name].get(k))) for k in ("w", "b")} if isinstance(raw[name], dict) else {}
        if shapes != {"w": (fi, fo), "b": (fo,)}:
            raise ValueError(f"{path}: {name} has shapes {shapes}, not w {(fi, fo)} / b {(fo,)} of the DeepMind 4x1024 net")


def init_params(seed: int, device="cuda") -> Dict[str, Dict[str, torch.Tensor]]:
    """Random-init weights of the architecture: haiku's default `hk.initializers.TruncatedNormal(stddev=1/sqrt(fan_in))`,
    i.e. a standard normal truncated to [-2, 2] by RESAMPLING (not clipping), scaled by 1/sqrt(fan_in); biases zero."""
    rng = np.random.default_rng(seed)
    out = {}
    for name, (fi, fo) in zip(LAYERS, SIZES):
        w = rng.normal(0, 1, (fi, fo))
        bad = np.abs(w) > 2
        while bad.any():  # rejection-resample the ~4.6 % of draws outside two sigma
            w[bad] = rng.normal(0, 1, int(bad.sum()))
            bad = np.abs(w) > 2
        w = w.astype(np.float32) / np.sqrt(fi).astype(np.float32)
        out[name] = {"w": torch.as_tensor(w, device=device), "b": torch.zeros(fo, dtype=torch.float32, device=device)}
    return out


def params_to_numpy(params) -> Dict[str, np.ndarray]:
    """flat {'w0'..'w5','b0'..'b5'} for the oracle's NumPy MLP"""
    flat = {}
    for i, name in enumerate(LAYERS):
        flat[f"w{i}"] = params[name]["w"].detach().cpu().numpy()
        flat[f"b{i}"] = params[name]["b"].detach().cpu().numpy()
    return flat


class PackedParams:
    """A net given as its packed blob (u8[brl_mlp_packed_bytes()], what `brl_mlp_pack` writes) instead of an fp32 parameter
    dict -- how a device-resident model zoo (zoo.ModelZoo) hands out an opponent.  Every ForwardPass method that takes
    `params` takes one: the forwards read the blob as is, and `pack_into` copies it (device to device)."""
    __slots__ = ("blob",)

    def __init__(self, blob: torch.Tensor):
        if blob.dtype != torch.uint8 or blob.dim() != 1 or blob.numel() != ops._lib.load().brl_mlp_packed_bytes():
            raise ValueError("PackedParams holds one packed blob: u8[brl_mlp_packed_bytes()]")
        self.blob = blob


class ForwardPass:
    """`hk.without_apply_rng(hk.transform(forward_fn))` look-alike: `.apply(params, x)`."""

    def __init__(self, activation: str = "relu", model_type: str = "DeepMind", precision: str = None):
        if model_type != "DeepMind":
            raise NotImplementedError("only the DeepMind 4x1024 net is on the hot path (SURVEY 8a a16)")
        if activation != "relu":  # all five bundled models and every ppo.py default are ReLU nets (src/models.py:28-31)
            raise NotImplementedError("the tensor-core forward fuses ReLU into its epilogues; tanh nets are not on the hot "
                                      "path (a cuBLAS forward for them: scripts/torch_baseline.TorchForwardPass)")
        if precision is None:
            precision = "tc"
        if precision not in ("tc", "tc-bf16"):
            raise ValueError(f"unknown precision {precision!r}: the product path has no library back end "
                             "(scripts/torch_baseline.py holds the cuBLAS cross-check)")
        self._activation = torch.relu
        self.precision = precision
        self._scratch = None
        self.seed_salt = None  # device int64[1] XORed into every sampling seed (set by a CUDA-graph rollout, see roll_out.py)

    @property
    def input_dtype(self):
        """dtype the forward consumes without a cast (env kernels can write the 0/1 observation in it directly)"""
        return torch.bfloat16

    def _packed(self, params):
        """bf16 hi/lo blob of `params`, re-packed when any tensor was replaced or updated in place."""
        if isinstance(params, PackedParams):
            return params.blob
        fixed = params.get("_brl_packed_fixed")  # a caller-owned blob at a fixed address (CUDA-graph rollout)
        if fixed is not None:
            return fixed
        ws = [params[name]["w"] for name in LAYERS]
        bs = [params[name]["b"] for name in LAYERS]
        stamp = tuple((t.data_ptr(), t._version) for t in ws + bs)
        cached = params.get("_brl_packed")
        if cached is None or cached[0] != stamp:
            cached = (stamp, ops.mlp_pack(ws, bs))
            params["_brl_packed"] = cached
        return cached[1]

    def _apply_tc(self, params, x: torch.Tensor):
        n = x.shape[0]
        xb = ops.obs_to_bf16(x.contiguous())
        self._ensure_scratch(n, x.device)
        logits = torch.empty((n, 38), dtype=torch.float32, device=x.device)
        value = torch.empty(n, dtype=torch.float32, device=x.device)
        ops.mlp_forward(xb, self._packed(params), self._scratch, logits, value, single_bf16=self.precision == "tc-bf16")
        return logits, value

    def act(self, params, x: torch.Tensor, mask, action: torch.Tensor, log_prob=None, value=None, *, sample: bool,
            seed: int, env_offset: int = 0):
        """`logits, value = apply(params, x)` followed by the masked categorical of src/roll_out.py:77-81 /
        src/utils.py:83-88, written into caller buffers.  The tensor-core precisions do it in one call
        (`brl_policy_act`: from 4096 envs on a single persistent launch with the sampler in the head epilogue)."""
        n = x.shape[0]
        xb = ops.obs_to_bf16(x.contiguous())
        self._ensure_scratch(n, x.device)
        ops.policy_act(xb, self._packed(params), self._scratch, mask, action, log_prob, value, sample=sample, seed=seed,
                       env_offset=env_offset, single_bf16=self.precision == "tc-bf16",
                       seed_salt=self.seed_salt if (sample and n >= 4096) else None)  # the salt lives in the fused launch

    def act_rows(self, params, obs_bf16: torch.Tensor, mask, action: torch.Tensor, rows: torch.Tensor, log_prob=None,
                 logits=None, *, sample: bool = False, seed: int = 0, env_offset: int = 0):
        """`act` for the envs listed in `rows` only (int32 indices into the full per-env arrays)."""
        n = rows.shape[0]
        if n == 0:
            return
        need = ops._lib.load().brl_mlp_rows_scratch_bytes(n)
        if self._scratch is None or self._scratch.numel() < need or self._scratch.device != obs_bf16.device:
            self._scratch = torch.empty(need, dtype=torch.uint8, device=obs_bf16.device)
        ops.policy_act_rows(obs_bf16, self._packed(params), self._scratch, mask, action, rows, log_prob, logits, sample=sample, seed=seed,
                            env_offset=env_offset, single_bf16=self.precision == "tc-bf16")

    def forward_into(self, params, obs_bf16: torch.Tensor, logits: torch.Tensor, value: torch.Tensor) -> None:
        """`apply` on a bf16 observation, written into caller buffers (f32 logits [n, 38], value [n]): one brl_mlp_forward.
        The roll-out records a KL anchor's logits with it."""
        self._ensure_scratch(obs_bf16.shape[0], obs_bf16.device)
        ops.mlp_forward(obs_bf16, self._packed(params), self._scratch, logits, value, single_bf16=self.precision == "tc-bf16")

    def pack_into(self, params, blob: torch.Tensor) -> torch.Tensor:
        """re-pack `params` into the caller's fixed-address blob (a PackedParams: a device-to-device copy of its blob)"""
        if isinstance(params, PackedParams):
            return blob.copy_(params.blob)
        return ops.mlp_pack([params[name]["w"] for name in LAYERS], [params[name]["b"] for name in LAYERS], out=blob)

    def _ensure_scratch(self, n, device):
        if self._scratch is None or self._scratch.numel() < ops._lib.load().brl_mlp_scratch_bytes(n) or \
                self._scratch.device != device:
            self._scratch = ops.mlp_scratch(n, device)

    def apply(self, params, x: torch.Tensor):
        return self._apply_tc(params, x)


def make_forward_pass(activation: str = "relu", model_type: str = "DeepMind", precision: str = None) -> ForwardPass:
    """src/models.py:73-83"""
    return ForwardPass(activation, model_type, precision)
