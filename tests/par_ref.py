"""Reference of the double-dummy par (DESIGN.md f13), restated without the device formulas.

Contracts are scored from the pinned reference scorer (tests/golden/score_table.npy) and IMPs converted with
tests/golden/imp_table.npy.  The par is found by plain memoised recursion over the competitive-bidding game, not by the
device's backward induction with suffix optima."""
import functools

import numpy as np

from tests import helpers as H

_SCORE = np.load(H.GOLDEN + "/score_table.npy")  # [bid, none/X/XX, vul, tricks]
_IMP = np.load(H.GOLDEN + "/imp_table.npy")      # IMPs of d = -8000..8000 step 10
PASSED_OUT = -1


def imp(d: int) -> int:
    """IMPs of an integer score difference (every score is a multiple of 10; 24 IMPs from 4000 on)"""
    d = max(-8000, min(8000, int(d)))
    return int(_IMP[(d + 8000) // 10])


def contract_score(bid: int, doubled: bool, vul: int, tricks: int) -> int:
    return int(_SCORE[bid, 1 if doubled else 0, int(vul), int(tricks)])


def declarer(dd, dealer: int, side: int, strain: int) -> int:
    """the partner of `side` with more tricks in `strain`; on a tie the one who comes first in the auction from the dealer"""
    a, b = side, side + 2
    if dd[a][strain] != dd[b][strain]:
        return a if dd[a][strain] > dd[b][strain] else b
    return a if (a - dealer) % 4 < (b - dealer) % 4 else b


def par(dd, dealer: int, vul_ns: int, vul_ew: int):
    """dd[seat][strain] (seats N,E,S,W; strains C,D,H,S,NT) -> (par in NS points, contract code): -1 when passed out,
    else bid | declarer_seat << 8 | doubled << 10"""
    dd = [[int(x) for x in row] for row in dd]
    vul = (int(vul_ns), int(vul_ew))

    def value(side, c):
        seat = declarer(dd, dealer, side, c % 5)
        t = dd[seat][c % 5]
        s = contract_score(c, t < c // 5 + 7, vul[side], t)
        return s if side == 0 else -s

    @functools.lru_cache(maxsize=None)
    def solve(owner, c, mover, passes):
        """(NS value, final (owner, contract) or None) with `mover` to call; pass is listed first, then contracts upward,
        and the first best option is taken"""
        if owner is None:
            options = [(0, None) if passes == 1 else solve(None, -1, 1 - mover, 1)]
        else:
            options = [(value(owner, c), (owner, c))]
        options += [solve(mover, c2, 1 - mover, 0) for c2 in range(c + 1, 35)]
        best = max(v for v, _ in options) if mover == 0 else min(v for v, _ in options)
        return next(o for o in options if o[0] == best)

    v, final = solve(None, -1, dealer % 2, 0)
    if final is None:
        return v, PASSED_OUT
    side, c = final
    seat = declarer(dd, dealer, side, c % 5)
    return v, c | seat << 8 | int(dd[seat][c % 5] < c // 5 + 7) << 10


def par_by_player(par_ns: int, seating) -> np.ndarray:
    """par in the rewards layout: by player id (p, p, -p, -p), p = par of the team of player ids {0, 1}; seating[seat] is the
    player id at that seat"""
    p = par_ns if int(seating[0]) >> 1 == 0 else -par_ns
    return np.array([p, p, -p, -p], dtype=np.float32)


def par_reward(score_actor: float, par_actor: float) -> np.float32:
    """the par_imp reward of a finished board: IMP(score - par) / 24 from the actor's side"""
    return np.float32(imp(int(score_actor) - int(par_actor))) / np.float32(24)
