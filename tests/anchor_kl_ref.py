"""TEST INFRASTRUCTURE ONLY: the KL-anchored PPO loss in float64 autograd, the reference the anchored CUDA loss head is
checked against.  loss = oracle/ppo_ref.loss_fn's total + anchor_kl_coef * mean_b KL(pi(.|s_b) || alpha(.|s_b)), with pi the
policy distribution of the loss (masked softmax, or the unmasked one) and alpha the anchor's softmax over the same
action set, both as log-softmax so that no term is log 0, and 0 log 0 := 0."""
from __future__ import annotations

import torch

from oracle import ppo_ref


def anchor_kl(logits, anchor_logits, mask, masked_policy=True):
    """mean_b KL(pi || alpha) over the policy's action set (the legal actions, or all of them)"""
    sel = mask if masked_policy else torch.ones_like(mask)
    neg_inf = torch.tensor(float("-inf"), dtype=logits.dtype)
    logp = torch.log_softmax(torch.where(sel, logits, neg_inf), dim=1)
    loga = torch.log_softmax(torch.where(sel, anchor_logits.to(logits.dtype), neg_inf), dim=1)
    p = torch.exp(logp)
    # the select comes BEFORE the product, so that autograd never sees 0 * (-inf - -inf)
    diff = torch.where(sel & (p > 0), logp - loga, torch.zeros_like(logp))
    return (p * diff).sum(1).mean()


def loss_fn(logits, value, mask, action, old_log_prob, old_value, gae, targets, *, anchor_logits=None, anchor_kl_coef=0.0,
            masked_policy=True, **kw):
    """ppo_ref.loss_fn, plus the KL term when anchor_logits is given -> (total, aux + (anchor_kl,))"""
    total, aux = ppo_ref.loss_fn(logits, value, mask, action, old_log_prob, old_value, gae, targets, masked_policy=masked_policy, **kw)
    if anchor_logits is None:
        return total, aux + (torch.zeros((), dtype=logits.dtype),)
    kl = anchor_kl(logits, anchor_logits, mask, masked_policy)
    return total + anchor_kl_coef * kl, aux + (kl,)
