"""TEST INFRASTRUCTURE ONLY (never imported by brl_b200/): CPU restatement of the supervised step of sl.py --
`loss` (sl.py:169-184) and `accuracy` (sl.py:186-194) in float64 PyTorch, with autograd standing in for
`jax.value_and_grad`, the test metrics (sl.py:288-301), optax.adam without clipping (sl.py:166) in NumPy, the
examples of make_dataset (sl.py:100-117) replayed on the C oracle -- and the data the tests and scripts/sl_bench.py
feed them: random-legal auctions played on the oracle, written in OpenSpiel's text format.

Parity status: the reference needs jax / haiku / optax / pyspiel, none installable here, so the loss and the optimizer
are pinned only by this restatement from the cited lines (as f1's ppo_ref.py); tests/test_sl_host.py checks it against
hand-worked answers.
"""
from __future__ import annotations

import numpy as np
import torch

from . import oracle as orc

NUM_ACTIONS = 38


def loss(logits, labels, legal, entropy_coef=0.0):
    """Returns (total_loss, (target_loss, entropy)) of sl.py:175-184.  `legal`: bool [B, 38]."""
    log_probs = torch.log_softmax(logits, dim=1)                                           # unmasked (sl.py:178)
    one_hot = torch.nn.functional.one_hot(labels.long(), NUM_ACTIONS).to(logits.dtype)
    target_loss = -(one_hot * log_probs).mean()                                            # over B * 38 entries (:179)
    # entropy of the policy over the legal calls, with the select semantics of SURVEY 7 (as ppo_ref.loss_fn)
    masked = torch.where(legal, logits, torch.tensor(float("-inf"), dtype=logits.dtype))
    logp = torch.log_softmax(masked, dim=1)
    entropy = -(torch.exp(logp) * torch.where(legal, logp, torch.zeros_like(logp))).sum(1).mean()   # :180-182
    return target_loss - entropy_coef * entropy, (target_loss, entropy)                    # :183-184


def accuracy(logits, labels):
    """sl.py:186-194: argmax of the unmasked softmax against the label (first index on ties)."""
    return (torch.softmax(logits, dim=1).argmax(dim=1) == labels.long()).to(logits.dtype).mean()


def test_metrics(logits, labels, legal, entropy_coef=0.0) -> dict:
    """sl.py:288-302 on one batch."""
    total, (target, entropy) = loss(logits, labels, legal, entropy_coef)
    pi = torch.softmax(logits, dim=1)
    return {"test/total_loss": float(total), "test/target_loss": float(target), "test/entropy": float(entropy),
            "test/test_accuracy": float(accuracy(logits, labels)),
            "test/illegal_actions_prob": float((pi * (~legal).to(pi.dtype)).sum(1).mean())}


def adam_step(p, g, m, v, count, *, lr, b1=0.9, b2=0.999, eps=1e-8):
    """One optax.adam(lr) step (eps 1e-8, no clipping) on flat float64 arrays; `count` = steps before this one."""
    g = np.asarray(g, np.float64)
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    t = count + 1
    return p - lr * (m / (1 - b1 ** t)) / (np.sqrt(v / (1 - b2 ** t)) + eps), m, v


def replay_examples(table, calls, offsets, traj, position, n_threads: int = 1):
    """make_dataset's example for each (trajectory, call position) on the C oracle: the env is placed on the trajectory's
    deal (dealer North, nobody vulnerable, players = seats), the calls before `position` are stepped, and the observation
    / legal mask of the player to act are read.  Examples are grouped by position so that every batch of oracle envs steps
    in lockstep.  Returns (obs u8 [B, 480], mask u8 [B, 38], label i32 [B])."""
    table = np.ascontiguousarray(table, dtype=np.uint8)
    traj = np.asarray(traj, dtype=np.int64)
    position = np.asarray(position, dtype=np.int64)
    offsets = np.asarray(offsets, dtype=np.int64)
    calls = np.asarray(calls)
    B = traj.shape[0]
    obs = np.zeros((B, orc.OBS_DIM), np.uint8)
    mask = np.zeros((B, orc.NUM_ACTIONS), np.uint8)
    label = calls[offsets[traj] + position].astype(np.int32)
    for p in np.unique(position):
        rows = np.flatnonzero(position == p)
        n = rows.shape[0]
        env = orc.OracleEnv(table, n, n_threads=n_threads)
        env.reset_fields(traj[rows], np.zeros(n), np.zeros(n), np.zeros(n), np.tile(np.arange(4, dtype=np.int8), (n, 1)))
        for k in range(int(p)):
            env.step(calls[offsets[traj[rows]] + k].astype(np.int32))
        out = env.export(np.uint8)
        obs[rows] = out["observation"]
        mask[rows] = out["legal_action_mask"]
    return obs, mask, label


def random_trajectories(n_traj: int, seed: int):
    """Random-legal auctions (dealer North, players = seats) played on the C oracle over synthetic deals."""
    from brl_b200.deals import synthetic_deal_table
    from brl_b200.sl import Trajectories
    table = synthetic_deal_table(n_traj, seed=seed)
    table[:, 32:] = 0
    env = orc.OracleEnv(table, n_traj)
    env.reset_fields(np.arange(n_traj), np.zeros(n_traj), np.zeros(n_traj), np.zeros(n_traj),
                     np.tile(np.arange(4, dtype=np.int8), (n_traj, 1)))
    calls = [[] for _ in range(n_traj)]
    for step in range(400):
        done = env.export()["terminated"].astype(bool)
        if done.all():
            break
        act = env.random_legal_actions(seed, step)
        for i in np.flatnonzero(~done):
            calls[i].append(int(act[i]))
        env.step(act)
    lens = np.array([len(c) for c in calls])
    return Trajectories(table=table, calls=np.concatenate(calls).astype(np.uint8),
                        offsets=np.concatenate([[0], np.cumsum(lens)]).astype(np.int64), line=np.arange(1, n_traj + 1))


def openspiel_lines(traj, rng):
    """Trajectories -> the ints of OpenSpiel lines: the deal in chance order (card at position k to seat k mod 4 from
    North), 52 + call, and a dummy 52-card play tail unless the deal is passed out."""
    from brl_b200.deals import unpack_deal_table
    owners = unpack_deal_table(traj.table)[0]
    out = []
    for i in range(len(traj)):
        chance = np.stack([rng.permutation(np.flatnonzero(owners[i] == s)) for s in range(4)], axis=1).reshape(-1)
        toks = np.concatenate([chance, traj.calls[traj.offsets[i]:traj.offsets[i + 1]].astype(np.int64) + 52])
        out.append(toks if len(toks) == 56 else np.concatenate([toks, rng.permutation(52)]))
    return out


def write_lines(path, lines) -> str:
    """Write lines of ints as the space-separated text sl.py reads."""
    with open(path, "w") as fh:
        fh.write("".join(" ".join(map(str, np.asarray(x, np.int64))) + "\n" for x in lines))
    return str(path)


def golden_lines(golden: dict):
    """the lines of tests/golden/sl_golden.npz"""
    return np.split(golden["line_ints"].astype(np.int64), np.cumsum(golden["line_len"])[:-1])
