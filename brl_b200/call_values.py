"""Which calls cost IMPs, and what a net should have called instead (DESIGN.md f16): host NumPy over the int64 sums of
`evaluation.make_call_values_evaluate` / `ops.call_values`.

What the numbers mean:
- A deviation (c, b -> a) of net m is the rule "in context c, when the net would call b, call a instead".  It conditions only
  on what the decider knows, and the continuation is the nets' own unchanged play, so its mean gain per decision estimates
  an implementable one-step change of the net's policy (in IMPs per decision, for the decider's team, the other table held
  at its result).
- A decision's regret maximises over the calls with the actual deal in hand: it is a hindsight upper bound on what any
  one call could have gained, not an achievable gain.
"""
from __future__ import annotations

from typing import Dict, List

import numpy as np

from .board_log import ACTION_STR
from .system import context_name


def _mean_se(n, s1, s2):
    """mean and standard error (ddof = 1) from {n, sum, sum of squares}, as float arrays (NaN where n < 2 for the SE)"""
    n = np.asarray(n, np.float64)
    mean = np.divide(s1, n, out=np.zeros_like(n), where=n > 0)
    var = np.divide(s2 - n * mean * mean, n - 1, out=np.full_like(n, np.nan), where=n > 1)
    se = np.sqrt(np.maximum(var, 0.0) / np.where(n > 1, n, 1))
    return mean, np.where(n > 1, se, np.nan)


class CallValues:
    """One net's sums: gain_sums [75, 38, 38, 4] and regret_sums [75, 4] ({n, sum, sum of squares, #(> 0)})."""

    def __init__(self, gain_sums, regret_sums, mismatch: int = 0):
        self.gain = np.asarray(gain_sums, np.int64)
        self.regret = np.asarray(regret_sums, np.int64)
        self.mismatch = int(mismatch)
        self.decisions = int(self.regret[:, 0].sum())

    def mean_regret(self) -> float:
        """regret per decision over all contexts (IMPs)"""
        return float(self.regret[:, 1].sum()) / self.decisions if self.decisions else 0.0

    def regret_table(self) -> List[Dict]:
        """per context with decisions: its name, decisions, mean regret, its SE and the share of decisions with regret > 0"""
        mean, se = _mean_se(self.regret[:, 0], self.regret[:, 1], self.regret[:, 2])
        return [dict(context=context_name(c), decisions=int(self.regret[c, 0]), mean_regret=float(mean[c]),
                     se=float(se[c]), share_positive=float(self.regret[c, 3]) / float(self.regret[c, 0]))
                for c in np.flatnonzero(self.regret[:, 0])]

    def top_deviations(self, k: int = 20, min_count: int = 30) -> List[Dict]:
        """the k deviations (c, b -> a), a != b, of largest total gain among those with at least `min_count` decisions and a
        positive mean: context, played, instead, decisions, mean gain ± SE (IMPs per decision) and total IMPs"""
        n, s1, s2 = (self.gain[..., j] for j in range(3))
        mean, se = _mean_se(n, s1, s2)
        ok = (n >= max(1, min_count)) & (mean > 0)
        ok &= ~np.eye(n.shape[1], dtype=bool)[None]
        cells = np.argwhere(ok)
        order = np.argsort(-s1[ok], kind="stable")[:k]
        return [dict(context=context_name(int(c)), played=ACTION_STR[b], instead=ACTION_STR[a], decisions=int(n[c, b, a]),
                     mean=float(mean[c, b, a]), se=float(se[c, b, a]), total_imps=int(s1[c, b, a]))
                for c, b, a in cells[order]]

    def summary(self, k: int = 20, min_count: int = 30) -> Dict:
        return dict(decisions=self.decisions, mean_regret=self.mean_regret(), mismatch=self.mismatch,
                    regret_by_context=self.regret_table(), top_deviations=self.top_deviations(k, min_count))


def from_sums(result: Dict) -> List[CallValues]:
    """one CallValues per net from make_call_values_evaluate's result"""
    return [CallValues(g, r, m) for g, r, m in zip(result["gain_sums"], result["regret_sums"], result["mismatch"])]


def compare(a: CallValues, b: CallValues) -> Dict:
    """b against a: the change of mean regret per decision overall and per context both nets decide in"""
    both = np.flatnonzero((a.regret[:, 0] > 0) & (b.regret[:, 0] > 0))
    ma = a.regret[both, 1] / a.regret[both, 0]
    mb = b.regret[both, 1] / b.regret[both, 0]
    return dict(mean_regret_change=b.mean_regret() - a.mean_regret(),
                by_context={context_name(int(c)): float(y - x) for c, x, y in zip(both, ma, mb)})
