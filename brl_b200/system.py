"""What a net's calls mean: reports over a bidding-system histogram (DESIGN.md f15).

A histogram hist[75, 38, 96] (one net of the int64 [M, 75, 38, 96] that `evaluation.make_bidding_system_evaluate`,
`ops.system_stats` or `from_auctions` produce) counts, per context and call, the hand behind each decision: columns 0..37
the HCP histogram, 38 + 14 * suit + length the suit-length histograms (clubs, diamonds, hearts, spades), 94 the balanced
hands, 95 the decisions.  The contexts are the first round of the auction:

    0..3     OPEN(p)        the opening decision in position p after the dealer (every earlier call Pass)
    4 + b    RESPONSE(b)    partner opened with bid b, right-hand opponent passed
    39 + b   OVERCALL(b)    right-hand opponent opened with bid b (the direct seat)
    74       OTHER          everything else

Everything here is host NumPy over a histogram, except `from_auctions`, which counts stored auctions on the device."""
from __future__ import annotations

from typing import Dict, List

import numpy as np

from .board_log import ACTION_STR

CONTEXTS, NUM_CALLS, COLS = 75, 38, 96
HCP, LEN, BAL, COUNT = slice(0, 38), 38, 94, 95
SUITS = ("C", "D", "H", "S")
OTHER = 74


def context_name(c: int) -> str:
    """OPEN(p), RESPONSE(1H), OVERCALL(1NT), OTHER"""
    if c < 4:
        return f"OPEN({c})"
    if c < 39:
        return f"RESPONSE({ACTION_STR[c - 4 + 3]})"
    if c < 74:
        return f"OVERCALL({ACTION_STR[c - 39 + 3]})"
    return "OTHER"


def response_context(bid: int) -> int:
    """RESPONSE(bid), bid 0..34 (1C .. 7NT)"""
    return 4 + bid


def overcall_context(bid: int) -> int:
    return 39 + bid


def _percentile(hist_row: np.ndarray, q: float) -> int:
    """the smallest HCP value whose cumulative share reaches q (-1 for an empty row)"""
    total = hist_row.sum()
    if total == 0:
        return -1
    return int(np.searchsorted(np.cumsum(hist_row), q * total - 1e-9))


class BiddingSystem:
    """Statistics of one net's histogram hist_m int[75, 38, 96]:
    - `frequency[c, a]`: the share of call a among the decisions in context c (0 where c has none);
    - per (c, a): `count`, `mean_hcp`, HCP percentiles `p10` / `p50` / `p90`, `mean_length[c, a, suit]` and `balanced`
      (the balanced share).  Means and shares are NaN and percentiles -1 where (c, a) has no decision."""

    def __init__(self, hist_m):
        h = np.asarray(hist_m, dtype=np.int64)
        if h.shape != (CONTEXTS, NUM_CALLS, COLS):
            raise ValueError(f"BiddingSystem: a histogram is int[{CONTEXTS}, {NUM_CALLS}, {COLS}], got {h.shape}")
        self.hist = h
        self.count = h[:, :, COUNT]
        per_context = self.count.sum(axis=1, keepdims=True)
        self.decisions = per_context[:, 0]
        with np.errstate(invalid="ignore", divide="ignore"):
            self.frequency = np.where(per_context > 0, self.count / np.maximum(per_context, 1), 0.0)
            n = self.count.astype(np.float64)
            self.mean_hcp = (h[:, :, HCP] * np.arange(38)).sum(axis=2) / n
            lens = h[:, :, LEN:LEN + 56].reshape(CONTEXTS, NUM_CALLS, 4, 14)
            self.mean_length = (lens * np.arange(14)).sum(axis=3) / n[:, :, None]
            self.balanced = h[:, :, BAL] / n
        self.p10, self.p50, self.p90 = (np.array([[_percentile(h[c, a, HCP], q) for a in range(NUM_CALLS)]
                                                  for c in range(CONTEXTS)]) for q in (0.1, 0.5, 0.9))

    def describe(self, context: int, min_share: float = 0.0) -> List[str]:
        """one text row per call made in `context` (share >= min_share), most frequent first, e.g.
        `1NT  31.4 %  HCP 15-17 (p10-p90), mean 16.1, balanced 93 %`"""
        rows = []
        for a in np.argsort(-self.frequency[context], kind="stable"):
            f = self.frequency[context, a]
            if self.count[context, a] == 0 or f < min_share:
                continue
            rows.append(f"{ACTION_STR[a]:<4} {100 * f:5.1f} %  HCP {self.p10[context, a]}-{self.p90[context, a]} (p10-p90), "
                        f"mean {self.mean_hcp[context, a]:.1f}, balanced {100 * self.balanced[context, a]:.0f} %")
        return rows

    def summary(self) -> Dict:
        """JSON-ready statistics of every context with decisions and of every call made there"""
        out = {}
        for c in np.flatnonzero(self.decisions):
            calls = {}
            for a in np.flatnonzero(self.count[c]):
                calls[ACTION_STR[a]] = dict(
                    count=int(self.count[c, a]), frequency=float(self.frequency[c, a]), mean_hcp=float(self.mean_hcp[c, a]),
                    hcp_p10=int(self.p10[c, a]), hcp_p50=int(self.p50[c, a]), hcp_p90=int(self.p90[c, a]),
                    mean_length=dict(zip(SUITS, map(float, self.mean_length[c, a]))), balanced=float(self.balanced[c, a]))
            out[context_name(int(c))] = dict(decisions=int(self.decisions[c]), calls=calls)
        return out


def compare(a: BiddingSystem, b: BiddingSystem) -> Dict:
    """How far system b is from system a: per context with decisions in both, the total-variation distance between the two
    call distributions and, per call both made there, mean_hcp(b) - mean_hcp(a); and `distance`, the contexts' TV distances
    weighted by their decisions in a and b together (0: the same calls everywhere, 1: disjoint)."""
    contexts, weights, tvs = {}, [], []
    for c in np.flatnonzero((a.decisions > 0) & (b.decisions > 0)):
        tv = 0.5 * float(np.abs(a.frequency[c] - b.frequency[c]).sum())
        both = np.flatnonzero((a.count[c] > 0) & (b.count[c] > 0))
        contexts[context_name(int(c))] = dict(
            tv=tv, hcp_shift={ACTION_STR[k]: float(b.mean_hcp[c, k] - a.mean_hcp[c, k]) for k in both})
        weights.append(int(a.decisions[c] + b.decisions[c]))
        tvs.append(tv)
    distance = float(np.average(tvs, weights=weights)) if weights else float("nan")
    return dict(distance=distance, contexts=contexts)


def from_auctions(traj_or_npz, device="cuda") -> BiddingSystem:
    """The system of stored auctions, counted on the device (brl_system_stats_auctions): an `sl.Trajectories` (deal rows in
    order, dealer North) or a mapping shaped like tests/golden/auctions.npz (`table` u8[n_deals, 48], `calls`, `offsets`
    [n + 1], optional `board` and `dealer` per auction)."""
    import torch

    from . import ops
    if hasattr(traj_or_npz, "calls") and hasattr(traj_or_npz, "table"):
        t = traj_or_npz
        table, calls, offsets, board, dealer = t.table, t.calls, t.offsets, None, None
    else:
        z = traj_or_npz
        table, calls, offsets = z["table"], z["calls"], z["offsets"]
        board = z["board"] if "board" in z else None
        dealer = z["dealer"] if "dealer" in z else None
    calls = np.asarray(calls)
    if calls.size and (calls.min() < 0 or calls.max() >= NUM_CALLS):
        raise ValueError("from_auctions: a call is outside 0..37")
    dev = torch.device(device)
    as_t = lambda x, dt: None if x is None else torch.as_tensor(np.asarray(x).astype(dt), device=dev)  # noqa: E731
    hist = ops.new_system_hist(1, dev)
    ops.system_stats_auctions(as_t(table, np.uint8), as_t(calls, np.uint8), as_t(offsets, np.int64), hist,
                              board=as_t(board, np.int32), dealer=as_t(dealer, np.int8))
    return BiddingSystem(ops.system_hist_counts(hist)[0].cpu().numpy())
