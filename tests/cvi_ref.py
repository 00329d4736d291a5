"""Call-value policy improvement (DESIGN.md f17) in float64 NumPy: the one reference for brl_cv_grad / brl_cv_eval.
Restates the definitions of include/brl_b200.h:

  legal    isfinite(g[b, a]) (brl_call_values' gains are NaN on illegal calls)
  pi       softmax of the logits over the legal calls; gbar = sum_a pi_a g_a; H = entropy of pi
  loss     -mean_b gbar_b / 24 - ent_coef * mean_b H_b
  grad     d loss / d l_j = -pi_j (g_j - gbar) / (24 B) + ent_coef * pi_j (log pi_j + H) / B (legal j), 0 otherwise
  stats    {loss, mean gbar, mean g of the argmax-logit legal call (lowest index on ties), mean (max g - that g), mean H,
            share of samples whose argmax-logit call has the maximal g, mean unmasked-softmax mass on illegal calls, 0}
A sample without a legal call adds 0 to every sum but the illegal mass (1).

`host_records_with_obs` is tests/call_values_ref.py's host loop with each decision's observation, the reference for the
training examples brl_call_values writes beside its records."""
import numpy as np

IMP_SCALE = 24.0


def _legal_softmax(logits, legal):
    z = np.where(legal, logits, -np.inf)
    mx = z.max(axis=1, keepdims=True)
    mx = np.where(np.isfinite(mx), mx, 0.0)
    e = np.where(legal, np.exp(z - mx), 0.0)
    s = e.sum(axis=1, keepdims=True)
    p = np.divide(e, s, out=np.zeros_like(e), where=s > 0)
    logp = np.where(legal & (p > 0), np.log(np.where(p > 0, p, 1.0)), 0.0)
    return p, logp


def loss_grad_stats(logits, gain, ent_coef=0.0):
    """(loss, dloss/dlogits [B, 38], stats[8]) in float64 for logits and gains [B, 38] (NaN: illegal)"""
    logits = np.asarray(logits, np.float64)
    gain = np.asarray(gain, np.float64)
    B = logits.shape[0]
    legal = np.isfinite(gain)
    any_legal = legal.any(axis=1)
    g = np.where(legal, gain, 0.0)
    p, logp = _legal_softmax(logits, legal)
    gbar = (p * g).sum(axis=1)
    H = -(p * logp).sum(axis=1)
    loss = -gbar.mean() / IMP_SCALE - ent_coef * H.mean()
    grad = np.where(legal, -p * (g - gbar[:, None]) / (IMP_SCALE * B) + ent_coef * p * (logp + H[:, None]) / B, 0.0)
    # the argmax-logit legal call, lowest index on ties (np.argmax returns the first maximum)
    arg = np.argmax(np.where(legal, logits, -np.inf), axis=1)
    g_arg = np.where(any_legal, g[np.arange(B), arg], 0.0)
    g_max = np.where(any_legal, np.where(legal, g, -np.inf).max(axis=1, initial=-np.inf), 0.0)
    hit = np.where(any_legal, g_arg == g_max, False)
    q = np.exp(logits - logits.max(axis=1, keepdims=True))
    q /= q.sum(axis=1, keepdims=True)
    ill = (q * ~legal).sum(axis=1)
    stats = np.array([loss, gbar.mean(), g_arg.mean(), (g_max - g_arg).mean(), H.mean(), hit.mean(), ill.mean(), 0.0])
    return loss, grad, stats


def torch_loss(logits, gain, ent_coef=0.0):
    """the loss as a float64 torch expression of `logits` (for autograd through the net); gain a float64 tensor"""
    import torch
    legal = torch.isfinite(gain)
    g = torch.where(legal, gain, torch.zeros_like(gain))
    z = torch.where(legal, logits, torch.full_like(logits, -torch.inf))
    logp = torch.log_softmax(z, dim=1)
    p = logp.exp()                                         # exactly 0 on illegal calls
    plogp = p * torch.where(legal, logp, torch.zeros_like(logp))  # no 0 * -inf, in the value or the gradient
    gbar = (p * g).sum(1)
    H = -plogp.sum(1)
    return -gbar.mean() / IMP_SCALE - ent_coef * H.mean()


def host_records_with_obs(env, nets, models, n, rng_key, precision="tc", tune=0):
    """tests/call_values_ref.host_records with each decision's observation: records["obs"] holds, record by record, the bits
    of the pre-step state's observation in bf16 (uint16 [., 480]; the 0/1 features are exact in bf16).  The host loop
    replays the match with duplicate_step once per base iteration, on the state whose live envs are that iteration's
    decisions in env order (the records' order), so the rows are read there, before the step updates the state in place."""
    import torch
    from brl_b200 import duplicate
    from tests import call_values_ref
    rows = []
    orig = duplicate.duplicate_step

    def recording(step_fn):
        inner = orig(step_fn)

        def step(state, action, table_a_info, table_b_info, **kw):
            live = torch.nonzero(state._terminated_u8 == 0).flatten()
            obs = state.observation[live].to(torch.bfloat16).view(torch.int16).cpu().numpy().view(np.uint16)
            rows.append(obs.reshape(-1, 480))
            return inner(state, action, table_a_info, table_b_info, **kw)
        return step

    duplicate.duplicate_step = recording   # host_records imports it at call time; the evaluators keep their own binding
    try:
        rec, R_a, R_b = call_values_ref.host_records(env, nets, models, n, rng_key, precision, tune)
    finally:
        duplicate.duplicate_step = orig
    rec["obs"] = np.concatenate(rows) if rows else np.zeros((0, 480), np.uint16)
    assert len(rec["obs"]) == len(rec["env"])
    return rec, R_a, R_b
