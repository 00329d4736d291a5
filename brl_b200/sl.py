"""Supervised bidding pre-training: `sl.py` of the reference (the recipe behind `model-sl.pkl`, the starting point of the
"RL after SL pretraining" models) on the B200-native path.

The data is OpenSpiel's bridge bidding text format (sl.py:87-97): one trajectory per line, space-separated ints -- 52
chance actions (the deal), every call as 52 + action, then 52 play actions.  A passed-out deal (exactly 56 ints) has no
play.  Examples are built on the GPU (`brl_sl_examples`: replay of a stored auction prefix with the env's own device
rules), and each step is `brl_sl_grad` (forward + cross-entropy head + backward on tcgen05), `brl_mlp_adam_step`
(optax.adam: eps 1e-8, no clipping) and `brl_sl_eval` on the same batch for the post-update train accuracy (sl.py:279).

Not mirrored: wandb (`log_fn` receives the same dicts), and `num_examples` / `output_samples` (sl.py:211-242), which prints
pyspiel state renderings of mispredicted auctions -- the config key is accepted and ignored.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Callable, Optional, Union

import numpy as np
import torch

from . import _lib
from . import deals as _deals
from . import ops
from .models import init_params, make_forward_pass
from .optim import flatten_params
from .ppo import save_params

NUM_CARDS = 52
NUM_PLAYERS = 4
MIN_ACTION = 52
NUM_ACTIONS = 38
METRIC_KEYS = ("train/total_loss", "train/target_loss", "train/entropy", "train/train_accuracy")
TEST_METRIC_KEYS = ("test/total_loss", "test/target_loss", "test/entropy", "test/test_accuracy", "test/illegal_actions_prob")


def default_config() -> dict:
    """SLConfig defaults (sl.py:52-81)."""
    return dict(iterations=400_000, train_batch=128, learning_rate=1e-4, eval_every=10_000, data_path=None, save_path=None,
                num_examples=3, eval_batch=10_000, rng_seed=42, entropy_coef=0.0, type_of_model="DeepMind", activation="relu")


def deal_owners(chance: np.ndarray) -> np.ndarray:
    """int[n, 52] chance actions (a deal) -> int8[n, 52] seat (0 N .. 3 W) holding each card.

    OpenSpiel deals the chance action at position k to the k-th seat after the dealer, k mod 4
    (workspace/test_bridge_with_openspiel.py:164-174), and the dealer of bridge(use_double_dummy_result=false) is North.
    The card index is the chance action itself, in the observation's rank * 4 + suit order (wb5/utils.py:18-26).  This is
    the only place that knows the convention (DESIGN.md section 5: unpinned, no OpenSpiel in the tree to check it against)."""
    chance = np.asarray(chance)
    owners = np.empty(chance.shape, dtype=np.int8)
    owners[np.arange(chance.shape[0])[:, None], chance] = np.arange(NUM_CARDS) % NUM_PLAYERS
    return owners


@dataclass
class Trajectories:
    """Auctions of a data file: deal table (deals.py rows, no double-dummy results), calls 0..37 of trajectory t at
    calls[offsets[t]:offsets[t + 1]], and the 1-based line of the file each trajectory came from."""
    table: np.ndarray
    calls: np.ndarray
    offsets: np.ndarray
    line: np.ndarray

    def __len__(self) -> int:
        return int(self.table.shape[0])

    def to(self, device) -> dict:
        return dict(table=torch.as_tensor(self.table, device=device), calls=torch.as_tensor(self.calls, device=device),
                    offsets=torch.as_tensor(self.offsets, device=device))


def parse_trajectories(path: str) -> Trajectories:
    """Parse and validate a data file on the host (no device check of the auctions; `load_trajectories` adds it).

    Mirrors `_no_play_trajectory` (sl.py:87-97): a line of exactly 56 ints is kept whole, any other line loses its last 52.
    Raises ValueError naming the line for a non-integer token, a trajectory with no call, a deal that is not a
    permutation of 0..51 or a call outside 52..89."""
    with open(path) as fh:
        rows = [ln.split() for ln in fh.read().split("\n")]
    lens = np.fromiter(map(len, rows), dtype=np.int64, count=len(rows))
    keep_line = np.flatnonzero(lens > 0)
    lens = lens[keep_line]
    line = keep_line + 1
    tokens = [t for r in rows for t in r]
    try:
        flat = np.array(tokens, dtype=np.int64)
    except ValueError:
        for ln, r in zip(line, (rows[i] for i in keep_line)):
            for t in r:
                try:
                    int(t)
                except ValueError:
                    raise ValueError(f"{path}:{ln}: not an integer: {t!r}") from None
        raise
    n = len(lens)
    keep = np.where(lens == NUM_CARDS + NUM_PLAYERS, lens, lens - NUM_CARDS)   # sl.py:94-97
    short = np.flatnonzero(keep <= NUM_CARDS)
    if len(short):
        raise ValueError(f"{path}:{line[short[0]]}: {lens[short[0]]} ints: no call after the 52 chance actions")
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]])
    deal = flat[starts[:, None] + np.arange(NUM_CARDS)]
    bad = np.flatnonzero((np.sort(deal, axis=1) != np.arange(NUM_CARDS)).any(axis=1))
    if len(bad):
        raise ValueError(f"{path}:{line[bad[0]]}: the first 52 ints are not a permutation of 0..51")
    line_of = np.repeat(np.arange(n), lens)
    pos = np.arange(flat.shape[0]) - starts[line_of]
    sel = (pos >= NUM_CARDS) & (pos < keep[line_of])
    calls = flat[sel] - MIN_ACTION
    bad = np.flatnonzero((calls < 0) | (calls >= NUM_ACTIONS))
    if len(bad):
        raise ValueError(f"{path}:{line[line_of[sel][bad[0]]]}: call {calls[bad[0]] + MIN_ACTION} outside 52..89")
    offsets = np.concatenate([[0], np.cumsum(keep - NUM_CARDS)]).astype(np.int64)
    table = _deals.pack_deal_table(deal_owners(deal), np.zeros((n, 4, 5), dtype=np.int64))
    return Trajectories(table=table, calls=calls.astype(np.uint8), offsets=offsets, line=line)


_STATUS = {_lib.SL_ILLEGAL: "an illegal call", _lib.SL_EARLY_END: "the auction ends before its last call",
           _lib.SL_NOT_ENDED: "the auction does not end with its last call"}


def check_trajectories(traj: Trajectories, device="cuda", path: str = "") -> None:
    """Replay every auction once on the device (brl_sl_examples check mode); raise ValueError naming the first bad line."""
    d = traj.to(device)
    status = torch.empty(len(traj), dtype=torch.uint8, device=device)
    ops.sl_check(d["table"], d["calls"], d["offsets"], status)
    st = status.cpu().numpy()
    bad = np.flatnonzero(st != _lib.SL_OK)
    if len(bad):
        raise ValueError(f"{path}:{traj.line[bad[0]]}: {_STATUS[int(st[bad[0]])]} ({len(bad)} bad trajectories)")


def load_trajectories(path: str, device="cuda") -> Trajectories:
    """`parse_trajectories` + the device check of every auction."""
    traj = parse_trajectories(path)
    check_trajectories(traj, device, path)
    return traj


class ShuffledStream:
    """The trajectory order of make_dataset (sl.py:103-106): endless passes over the file, each a fresh shuffle, one
    example per trajectory per pass; a batch may straddle two passes.  (The call position of each example is drawn on the
    device, brl_sl_examples.)"""

    def __init__(self, n: int, seed: int):
        self.n = int(n)
        self.rng = np.random.default_rng(seed)
        self.perm = self.rng.permutation(self.n)
        self.pos = 0

    def take(self, k: int) -> np.ndarray:
        out = np.empty(k, dtype=np.int32)
        got = 0
        while got < k:
            if self.pos == self.n:
                self.perm = self.rng.permutation(self.n)
                self.pos = 0
            m = min(k - got, self.n - self.pos)
            out[got:got + m] = self.perm[self.pos:self.pos + m]
            got += m
            self.pos += m
        return out


def _metrics(prefix: str, s: np.ndarray, accuracy: float) -> dict:
    out = {f"{prefix}/total_loss": float(s[0]), f"{prefix}/target_loss": float(s[1]), f"{prefix}/entropy": float(s[2]),
           f"{prefix}/{prefix}_accuracy": accuracy}
    if prefix == "test":
        out["test/illegal_actions_prob"] = float(s[4])
    return out


def train(config: dict, data_path: Optional[str] = None, train: Union[None, str, Trajectories] = None,
          test: Union[None, str, Trajectories] = None, device="cuda", log_fn: Optional[Callable[[dict], None]] = None):
    """`main()` of sl.py:148-311.  `train` / `test`: Trajectories or file paths; default `data_path` (argument, else
    config["data_path"]) / {train,test}.txt.  `log_fn(metrics)` is called once per step, in order, with the keys of
    sl.py:280-285 (plus sl.py:296-302's test metrics on every `eval_every`-th step).  Checkpoints:
    save_path/params-{step}.pkl (sl.py:303-307), loadable by models.load_params.  Returns the parameters (haiku layout).

    Per-step statistics stay in a device buffer and are read once per `eval_every` block: the loop never waits for the
    device inside a block."""
    cfg = default_config()
    cfg.update(config)
    make_forward_pass(cfg["activation"], cfg["type_of_model"])  # FAIR / tanh nets raise, as everywhere on the hot path
    dev = torch.device(device)
    data_path = data_path or cfg["data_path"]

    def as_traj(x, name):
        if x is None:
            if data_path is None:
                raise ValueError(f"sl.train: no {name} data (pass {name}= or data_path)")
            x = os.path.join(data_path, f"{name}.txt")
        return load_trajectories(x, dev) if isinstance(x, str) else x

    train_t, test_t = as_traj(train, "train"), as_traj(test, "test")
    B, EB, every = int(cfg["train_batch"]), int(cfg["eval_batch"]), int(cfg["eval_every"])
    lr, ent = float(cfg["learning_rate"]), float(cfg["entropy_coef"])
    seed = int(cfg["rng_seed"])
    params = init_params(seed, dev)                                   # sl.py:267-268
    flat, views = flatten_params(params)
    blob = ops.mlp_pack_train(flat)
    m, v = torch.zeros_like(flat), torch.zeros_like(flat)
    grads = torch.empty_like(flat)
    scratch = ops.mlp_train_scratch(max(B, EB), dev)                   # each call lays out its own batch inside
    dtr, dte = train_t.to(dev), test_t.to(dev)
    obs = torch.empty((B, ops.OBS_DIM), dtype=torch.uint8, device=dev)
    mask = torch.empty((B, NUM_ACTIONS), dtype=torch.uint8, device=dev)
    label = torch.empty(B, dtype=torch.int32, device=dev)
    tobs = torch.empty((EB, ops.OBS_DIM), dtype=torch.uint8, device=dev)
    tmask = torch.empty((EB, NUM_ACTIONS), dtype=torch.uint8, device=dev)
    tlabel = torch.empty(EB, dtype=torch.int32, device=dev)
    acc_g, acc_e = ops.sl_acc(dev), ops.sl_acc(dev)
    stream_tr, stream_te = ShuffledStream(len(train_t), seed), ShuffledStream(len(test_t), seed + 1)
    # positions: Philox keyed by (seed, step, example); the test set uses its own key
    seed_tr, seed_te = seed, seed ^ 0x5445535453455430
    iterations = int(cfg["iterations"])
    stats = torch.zeros((min(every, iterations) if iterations else 1, 2, 8), dtype=torch.float32, device=dev)
    tstats = torch.zeros(8, dtype=torch.float32, device=dev)
    step = 0
    while step < iterations:
        k_steps = min(every - step % every, iterations - step)
        idx = torch.from_numpy(stream_tr.take(k_steps * B)).pin_memory().to(dev, non_blocking=True)
        for k in range(k_steps):
            s = step + k
            ops.sl_examples(dtr["table"], dtr["calls"], dtr["offsets"], idx[k * B:(k + 1) * B], obs, mask, label,
                            seed=seed_tr, step=s)
            ops.sl_grad(obs, blob, scratch, mask, label, grads, stats[k, 0], acc_g, ent_coef=ent)
            ops.mlp_adam_step(flat, grads, m, v, acc_g[14:15], blob, step=s + 1, lr=lr, eps=1e-8, max_grad_norm=0.0)
            ops.sl_eval(obs, blob, scratch, mask, label, stats[k, 1], acc_e, ent_coef=ent)   # sl.py:279, after the update
        step += k_steps
        test_metrics = None
        if step % every == 0:                                                                 # sl.py:288-309
            tidx = torch.from_numpy(stream_te.take(EB)).to(dev)
            ops.sl_examples(dte["table"], dte["calls"], dte["offsets"], tidx, tobs, tmask, tlabel, seed=seed_te,
                            step=step // every - 1)
            ops.sl_eval(tobs, blob, scratch, tmask, tlabel, tstats, acc_e, ent_coef=ent)
            ts = tstats.cpu().numpy()
            test_metrics = _metrics("test", ts, float(ts[3]))
            if cfg["save_path"] is not None:
                os.makedirs(cfg["save_path"], exist_ok=True)
                save_params(views, os.path.join(cfg["save_path"], f"params-{step}.pkl"))
        host = stats[:k_steps].cpu().numpy()
        if log_fn is not None:
            for k in range(k_steps):
                metrics = _metrics("train", host[k, 0], float(host[k, 1, 3]))
                if test_metrics is not None and k == k_steps - 1:
                    metrics.update(test_metrics)
                log_fn(metrics)
    return views
