"""The bidding-system statistics (DESIGN.md f15) in plain Python: the one reference for brl_system_stats and
brl_system_stats_auctions.  Restates the definitions next to `contract_score` / `par_score` in csrc/env_device.cuh:

  context of call t (call k made by seat (dealer + k) mod 4), from the earlier calls c_0 .. c_{t-1}:
    t        OPEN(t)       every earlier call is Pass
    4 + b    RESPONSE(b)   the only bid so far is b, made by the caller's partner at call t - 2; call t - 1 was Pass; no X / XX
    39 + b   OVERCALL(b)   the only bid so far is b, made by the caller's right-hand opponent at call t - 1
    74       OTHER
  hand features: HCP (A 4, K 3, Q 2, J 1), suit lengths (clubs, diamonds, hearts, spades), balanced (no void or singleton,
  at most one doubleton)
  hist[M, 75, 38, 96]: columns 0..37 HCP, 38 + 14 suit + len suit lengths, 94 balanced, 95 decisions."""
import numpy as np

CONTEXTS, COLS, OTHER = 75, 96, 74
NUM_ACTIONS = 38


def context(calls, t: int) -> int:
    """context of call t of `calls` (0 Pass, 1 X, 2 XX, 3 + bid)"""
    earlier = [int(c) for c in calls[:t]]
    bids = [k for k, c in enumerate(earlier) if c >= 3]
    if not bids:
        return t if t < 4 else OTHER
    if len(bids) > 1 or any(c in (1, 2) for c in earlier):
        return OTHER
    k, b = bids[0], earlier[bids[0]] - 3
    if k == t - 1:
        return 39 + b
    if k == t - 2 and earlier[t - 1] == 0:
        return 4 + b
    return OTHER


def hand_features(owners, seat: int):
    """(hcp, [len clubs, diamonds, hearts, spades], balanced) of `seat` from owners[52] (card c = rank * 4 + suit)"""
    cards = [c for c in range(52) if int(owners[c]) == seat]
    hcp = sum(max(0, c // 4 - 8) for c in cards)          # rank 9 J .. 12 A -> 1 .. 4
    lens = [sum(1 for c in cards if c % 4 == s) for s in range(4)]
    balanced = min(lens) >= 2 and sum(1 for x in lens if x == 2) <= 1
    return hcp, lens, balanced


def add_call(hist, owners, dealer: int, calls, t: int, net: int) -> None:
    """hist[M, 75, 38, 96] (int64) += call t of an auction, for net `net`"""
    hcp, lens, balanced = hand_features(owners, (dealer + t) % 4)
    row = hist[net, context(calls, t), int(calls[t])]
    row[hcp] += 1
    for s in range(4):
        row[38 + 14 * s + lens[s]] += 1
    row[94] += int(balanced)
    row[95] += 1


def add_auction(hist, owners, dealer: int, calls, net_of_seat=(0, 0, 0, 0)) -> None:
    """hist[M, 75, 38, 96] (int64) += every call of one auction, each for net net_of_seat[seat of the caller]"""
    for t in range(len(calls)):
        add_call(hist, owners, dealer, calls, t, net_of_seat[(dealer + t) % 4])


def new_hist(n_models: int = 1):
    return np.zeros((n_models, CONTEXTS, NUM_ACTIONS, COLS), dtype=np.int64)


def auctions_hist(owners_table, calls, offsets, board=None, dealer=None):
    """int64 [1, 75, 38, 96] of stored auctions: auction t is calls[offsets[t]:offsets[t + 1]] on owners_table[board[t]]
    (None: row t) with dealer dealer[t] (None: North)"""
    hist = new_hist(1)
    for t in range(len(offsets) - 1):
        row = t if board is None else int(board[t])
        d = 0 if dealer is None else int(dealer[t])
        add_auction(hist, owners_table[row], d, calls[int(offsets[t]):int(offsets[t + 1])])
    return hist
