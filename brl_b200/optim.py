"""Optimizer of ppo.py:186-211: `optax.chain(optax.clip_by_global_norm(max_grad_norm),
optax.adam(lr, eps=1e-5))`, with the optional linear learning-rate schedule, over ONE flat
fp32 parameter buffer (one fused sum-of-squares + one fused Adam kernel per step)."""
from __future__ import annotations

from typing import Callable, Dict, NamedTuple, Optional, Union

import torch

from . import ops
from .models import LAYERS


def flatten_params(params, clone: bool = True, out: Optional[torch.Tensor] = None):
    """-> (flat fp32 buffer, params dict whose tensors are views into it, in LAYERS order w then b).  `out`: the flat
    buffer to fill (e.g. one learner's row of a stacked population buffer) instead of a new one."""
    tensors = [params[name][k] for name in LAYERS for k in ("w", "b")]
    n = sum(t.numel() for t in tensors)
    flat = torch.empty(n, dtype=torch.float32, device=tensors[0].device) if out is None else out
    out, off = {}, 0
    for name in LAYERS:
        out[name] = {}
        for k in ("w", "b"):
            t = params[name][k]
            view = flat[off: off + t.numel()].view(t.shape)
            view.copy_(t.detach())
            out[name][k] = view
            off += t.numel()
    return flat, out


class OptState(NamedTuple):
    """optax's (EmptyState, ScaleByAdamState(count, mu, nu)) as flat buffers."""
    count: int
    mu: torch.Tensor
    nu: torch.Tensor


class AdamWithClip:
    def __init__(self, learning_rate: Union[float, Callable[[int], float]], eps: float = 1e-5, b1: float = 0.9,
                 b2: float = 0.999, max_grad_norm: Optional[float] = None):
        self.learning_rate, self.eps, self.b1, self.b2 = learning_rate, eps, b1, b2
        self.max_grad_norm = float(max_grad_norm) if max_grad_norm else 0.0
        self._scratch: Dict[torch.device, torch.Tensor] = {}

    def init(self, params) -> OptState:
        n = sum(params[name][k].numel() for name in LAYERS for k in ("w", "b"))
        dev = params[LAYERS[0]]["w"].device
        return OptState(0, torch.zeros(n, dtype=torch.float32, device=dev), torch.zeros(n, dtype=torch.float32, device=dev))

    def lr_at(self, count: int) -> float:
        """optax evaluates a schedule at the count BEFORE the increment."""
        return float(self.learning_rate(count)) if callable(self.learning_rate) else float(self.learning_rate)

    def update_(self, flat_params: torch.Tensor, flat_grads: torch.Tensor, state: OptState, sumsq=None) -> OptState:
        """In place on `flat_params`, `state.mu`, `state.nu`; returns the advanced state.  `sumsq`: f64[1] sum of squares of
        `flat_grads` when the producer of the gradient already formed it (ops.ppo_grad)."""
        scratch = self._scratch.get(flat_params.device)
        if scratch is None:
            scratch = self._scratch[flat_params.device] = torch.zeros(1, dtype=torch.float64, device=flat_params.device)
        ops.adam_clip(flat_params, flat_grads, state.mu, state.nu, scratch, step=state.count + 1, lr=self.lr_at(state.count),
                      beta1=self.b1, beta2=self.b2, eps=self.eps, max_grad_norm=self.max_grad_norm, sumsq=sumsq)
        return OptState(state.count + 1, state.mu, state.nu)


    def update_mlp_(self, flat_params, flat_grads, state: OptState, sumsq, blob) -> OptState:
        """`update_` for the flat DeepMind-MLP parameters with `ops.ppo_grad`'s sum of squares, refreshing the training
        blob in the same kernel pass (brl_mlp_adam_step)."""
        ops.mlp_adam_step(flat_params, flat_grads, state.mu, state.nu, sumsq, blob, step=state.count + 1, lr=self.lr_at(state.count),
                          beta1=self.b1, beta2=self.b2, eps=self.eps, max_grad_norm=self.max_grad_norm)
        return OptState(state.count + 1, state.mu, state.nu)


def update_mlp_grouped_(optimizers, flat_params, flat_grads, m, v, states, acc, blob):
    """`AdamWithClip.update_mlp_` for K learners in one launch (ops.mlp_adam_step_grouped): flat_params / flat_grads / m /
    v float32[K, ops.mlp_param_stride()] with states[k].mu / .nu = m[k, :n] / v[k, :n], acc the float64[K, ...] scratch of `ops.ppo_grad_grouped`, blob
    uint8[K, ...].  Each learner steps with its own optimizer's learning rate (schedule), clipping, betas and eps.
    Returns the advanced states."""
    ops.mlp_adam_step_grouped(flat_params, flat_grads, m, v, acc, blob, steps=[st.count + 1 for st in states],
                              lrs=[o.lr_at(st.count) for o, st in zip(optimizers, states)],
                              max_grad_norms=[o.max_grad_norm for o in optimizers], beta1=[o.b1 for o in optimizers],
                              beta2=[o.b2 for o in optimizers], eps=[o.eps for o in optimizers])
    return [OptState(st.count + 1, st.mu, st.nu) for st in states]


def make_optimizer(config) -> AdamWithClip:
    """ppo.py:186-211 from the same config keys."""
    lr = config["lr"]
    if config.get("anneal_lr", False):
        nmb, ep, nu = config["num_minibatches"], config["update_epochs"], config["num_updates"]
        base = lr

        def lr(count):  # noqa: F811 -- linear_schedule, ppo.py:186-192
            return base * (1.0 - (count // (nmb * ep)) / nu)
    clip = config["max_grad_norm"] if config.get("global_gradient_clipping", True) else None
    return AdamWithClip(lr, eps=1e-5, max_grad_norm=clip)
