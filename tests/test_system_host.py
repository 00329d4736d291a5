"""CPU: the bidding-system statistics (DESIGN.md f15) -- the reference's contexts on hand-built auctions and its hand features
on hand-built hands, the report (brl_b200/system.py) on a hand-made histogram, the ops' registration and the wrappers'
argument checks before any device work, and scripts/bidding_system.py's arguments."""
import numpy as np
import pytest
import torch

from tests import system_ref as R

P, X, XX = 0, 1, 2


def bid(level, strain):  # strain 0 C .. 4 NT
    return 3 + 5 * (level - 1) + strain


def test_contexts_of_hand_built_auctions():
    one_nt, two_c, one_h, one_c, one_s = bid(1, 4), bid(2, 0), bid(1, 2), bid(1, 0), bid(1, 3)
    calls = [one_nt, P, two_c, P]                                  # dealer N: 1NT P 2C P
    assert [R.context(calls, t) for t in range(4)] == [0, 39 + one_nt - 3, 4 + one_nt - 3, R.OTHER]
    assert R.context([P, one_h, X], 2) == 39 + one_h - 3           # P 1H X: the X is OVERCALL(1H)
    assert R.context([P, one_h, X], 1) == 1                        # third call of nothing: OPEN(1)
    assert R.context([one_c, one_s, P], 2) == R.OTHER              # two bids
    assert R.context([P, P, P], 3) == 3                            # fourth seat
    assert R.context([one_c, X, P], 3) == R.OTHER                  # a double before the response
    assert R.context([one_c, P, P], 3) == R.OTHER                  # balancing seat: partner's bid three calls back
    assert R.context([one_c, P, P, X], 4) == R.OTHER


def _owners(hands):
    """owners[52] from {seat: list of (rank, suit)}; the other cards go to the other seats in turn"""
    owners = np.full(52, -1, dtype=np.int8)
    for seat, cards in hands.items():
        for rank, suit in cards:
            owners[rank * 4 + suit] = seat
    free = [s for s in range(4) if s not in hands]
    rest = np.flatnonzero(owners < 0)
    for k, c in enumerate(rest):
        owners[c] = free[k // 13]
    return owners


def _hand(lengths, top=True):
    """a hand with these suit lengths (C, D, H, S): the highest cards of each suit (top) or the lowest"""
    return [(12 - r if top else r, s) for s, n in enumerate(lengths) for r in range(n)]


@pytest.mark.parametrize("shape,balanced", [((3, 3, 3, 4), True), ((2, 4, 4, 3), True), ((3, 5, 3, 2), True),
                                            ((5, 4, 2, 2), False), ((1, 4, 4, 4), False), ((6, 3, 3, 1), False),
                                            ((0, 4, 4, 5), False), ((7, 2, 2, 2), False)])
def test_hand_features_of_shapes(shape, balanced):
    hcp, lens, bal = R.hand_features(_owners({0: _hand(shape, top=False)}), 0)
    assert lens == list(shape) and bal == balanced and hcp == 0


def test_hand_features_of_hcp_extremes():
    top = [(r, s) for r in (12, 11, 10) for s in range(4)] + [(9, 0)]     # AKQ of every suit and the jack of clubs
    assert R.hand_features(_owners({2: top}), 2)[0] == 37
    assert R.hand_features(_owners({1: _hand((4, 3, 3, 3), top=False)}), 1)[0] == 0
    o = _owners({3: [(12, 0), (11, 1), (10, 2), (9, 3)] + [(r, s) for r in range(3) for s in range(3)]})
    assert R.hand_features(o, 3)[0] == 10


def test_reference_histogram_of_one_auction():
    owners = _owners({0: _hand((3, 3, 3, 4)), 2: _hand((5, 4, 2, 2), top=False)})
    h = R.new_hist(2)
    calls = [bid(1, 4), P, bid(2, 0), P, P, P]
    R.add_auction(h, owners, 0, calls, net_of_seat=(0, 1, 0, 1))
    row = h[0, 0, bid(1, 4)]                                       # N's 1NT opening, net 0
    assert row[95] == 1 and row[94] == 1 and row[R.hand_features(owners, 0)[0]] == 1
    assert [row[38 + 14 * s + n] for s, n in enumerate((3, 3, 3, 4))] == [1, 1, 1, 1]
    assert h[0, 4 + bid(1, 4) - 3, bid(2, 0), 95] == 1             # S's 2C response, net 0
    assert h[1, 39 + bid(1, 4) - 3, P, 95] == 1                    # E's pass over 1NT, net 1
    assert h[:, :, :, 95].sum() == len(calls) and h[1, :, :, 95].sum() == 3


def _hand_made_hist():
    """context OPEN(0): 1NT three times (HCP 15, 16, 17, balanced twice), Pass once (HCP 5); context 4 + 2 (RESPONSE(1H)): 2C once"""
    from brl_b200 import system
    h = np.zeros((system.CONTEXTS, system.NUM_CALLS, system.COLS), dtype=np.int64)
    nt = bid(1, 4)
    for hcp, shape, bal in ((15, (4, 3, 3, 3), 1), (16, (4, 4, 3, 2), 1), (17, (5, 4, 3, 1), 0)):
        h[0, nt, hcp] += 1
        for s, n in enumerate(shape):
            h[0, nt, 38 + 14 * s + n] += 1
        h[0, nt, 94] += bal
        h[0, nt, 95] += 1
    h[0, P, 5] += 1
    for s, n in enumerate((4, 3, 3, 3)):
        h[0, P, 38 + 14 * s + n] += 1
    h[0, P, 94] += 1
    h[0, P, 95] += 1
    h[6, bid(2, 0), 10] += 1
    h[6, bid(2, 0), 95] += 1
    return h


def test_report_statistics_of_a_hand_made_histogram():
    from brl_b200 import system
    s = system.BiddingSystem(_hand_made_hist())
    nt = bid(1, 4)
    assert s.decisions[0] == 4 and s.frequency[0, nt] == 0.75 and s.frequency[0, P] == 0.25
    assert s.count[0, nt] == 3 and s.mean_hcp[0, nt] == 16.0
    assert (s.p10[0, nt], s.p50[0, nt], s.p90[0, nt]) == (15, 16, 17)
    assert np.allclose(s.mean_length[0, nt], [13 / 3, 11 / 3, 3.0, 2.0])
    assert np.isclose(s.balanced[0, nt], 2 / 3)
    assert np.isnan(s.mean_hcp[0, 5]) and s.p50[0, 5] == -1 and s.frequency[1].sum() == 0
    rows = s.describe(0)
    assert rows[0] == "1NT   75.0 %  HCP 15-17 (p10-p90), mean 16.0, balanced 67 %" and rows[1].startswith("Pass  25.0 %")
    summ = s.summary()
    assert set(summ) == {"OPEN(0)", "RESPONSE(1H)"} and summ["OPEN(0)"]["calls"]["1NT"]["hcp_p50"] == 16
    assert system.context_name(4 + 2) == "RESPONSE(1H)" and system.context_name(39 + 34) == "OVERCALL(7NT)"
    # the same system is at distance 0; moving every 1NT opening to Pass gives TV 0.75 there
    assert system.compare(s, s)["distance"] == 0.0
    h2 = _hand_made_hist()
    h2[0, P] += h2[0, nt]
    h2[0, nt] = 0
    c = system.compare(s, system.BiddingSystem(h2))
    assert c["contexts"]["OPEN(0)"]["tv"] == 0.75 and c["contexts"]["RESPONSE(1H)"]["tv"] == 0.0
    assert np.isclose(c["distance"], 0.75 * 8 / 10)
    assert c["contexts"]["OPEN(0)"]["hcp_shift"] == {"Pass": (5 + 15 + 16 + 17) / 4 - 5}
    with pytest.raises(ValueError):
        system.BiddingSystem(np.zeros((75, 38, 95)))


def test_ops_are_registered_with_their_xla_layouts():
    from brl_b200 import _lib
    L = _lib.load()
    for name in ("brl_system_stats", "brl_system_stats_auctions"):
        assert name in _lib.OPS and name in _lib.LAZY_OPS and name + "_xla" in _lib.XLA_LEGACY
        assert L.brl_xla_layout(name.encode()) == b"iiiiix"
    assert L.brl_xla_layout(b"brl_duplicate_match") == b"iiiiisoxooooooooooooo"


def test_wrappers_check_their_arguments_before_any_device_work():
    from brl_b200 import _lib, ops
    n = 10
    state, table = torch.zeros((5, n, 4), dtype=torch.int32), torch.zeros((100, 48), dtype=torch.uint8)
    action, hist = torch.zeros(n, dtype=torch.int32), torch.zeros((2, 75, 38, 96), dtype=torch.uint32)
    with pytest.raises(_lib.BrlError, match="u32"):
        ops.system_stats(state, table, action, torch.zeros((2, 75, 38, 95), dtype=torch.uint32))
    with pytest.raises(_lib.BrlError, match="u32"):
        ops.system_stats(state, table, action, hist.to(torch.int64))
    with pytest.raises(_lib.BrlError, match="env_models"):
        ops.system_stats(state, table, action, hist, env_models=torch.zeros((n, 3), dtype=torch.int32))
    with pytest.raises(_lib.BrlError, match="done"):
        ops.system_stats(state, table, action, hist, done=torch.zeros(n + 1, dtype=torch.uint8))
    with pytest.raises(_lib.BrlError, match="packed state"):
        ops.system_stats(state[:, :5], table, action, hist)
    with pytest.raises(_lib.BrlError, match="CUDA"):      # every shape right: the first thing left is the device
        ops.system_stats(state, table, action, hist)
    calls, offsets, one = torch.tensor([0, 0, 0, 0], dtype=torch.uint8), torch.tensor([0, 4], dtype=torch.int64), hist[:1]
    with pytest.raises(_lib.BrlError, match=r"u32 \[1"):
        ops.system_stats_auctions(table, calls, offsets, hist)
    with pytest.raises(_lib.BrlError, match="outside 0..37"):
        ops.system_stats_auctions(table, torch.tensor([0, 38, 0, 0], dtype=torch.uint8), offsets, one)
    with pytest.raises(_lib.BrlError, match="rise"):
        ops.system_stats_auctions(table, calls, torch.tensor([0, 5], dtype=torch.int64), one)
    with pytest.raises(_lib.BrlError, match="board row"):
        ops.system_stats_auctions(table, calls, offsets, one, board=torch.tensor([100], dtype=torch.int32))
    with pytest.raises(_lib.BrlError, match="dealer is outside"):
        ops.system_stats_auctions(table, calls, offsets, one, dealer=torch.tensor([4], dtype=torch.int8))
    with pytest.raises(_lib.BrlError, match="int8"):
        ops.system_stats_auctions(table, calls, offsets, one, dealer=torch.tensor([0], dtype=torch.int32))
    with pytest.raises(_lib.BrlError, match="CUDA"):
        ops.system_stats_auctions(table, calls, offsets, one)
    ops.system_stats_auctions(table, calls[:0], torch.zeros(1, dtype=torch.int64), one)   # no auctions: nothing to do
    keys, pool = torch.zeros(n, dtype=torch.int64), torch.zeros((2, ops.mlp_pool_stride()), dtype=torch.uint8)
    scratch = torch.zeros(ops.duplicate_match_scratch_bytes(n, 2), dtype=torch.uint8)
    with pytest.raises(_lib.BrlError, match=r"u32 \[2"):
        ops.duplicate_match(keys, table, pool, scratch, torch.zeros(n), torch.zeros(8, dtype=torch.float64),
                            torch.zeros(1, dtype=torch.int32), system_hist=hist[:1])


def test_the_device_ops_check_their_buffers():
    import ctypes
    from brl_b200 import _lib
    L = _lib.load()
    for name in ("brl_system_stats", "brl_system_stats_auctions"):
        fn = getattr(L, name)
        fn.restype, fn.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]
        p0 = _lib.BrlParams(0, 0, 0, 0, 100, 0, 0, 1, -1.0, 1.0, 0.0, 0.0)
        assert fn(None, (ctypes.c_void_p * 6)(), ctypes.byref(p0), ctypes.sizeof(p0)) == 0       # an empty batch: a no-op
        p = _lib.BrlParams(10, 0, 0, 0, 100, 0, 0, 1, -1.0, 1.0, 0.0, 0.0)
        assert fn(None, (ctypes.c_void_p * 6)(4096, 4096, 4096, None, None, None), ctypes.byref(p), ctypes.sizeof(p)) == -2
        assert b"hist" in L.brl_last_error()
    fn = L.brl_system_stats
    p = _lib.BrlParams(10, 0, 0, 0, 100, 0, 0, 0, -1.0, 1.0, 0.0, 0.0)                   # k_steps = M = 0
    assert fn(None, (ctypes.c_void_p * 6)(*[4096] * 6), ctypes.byref(p), ctypes.sizeof(p)) == -1
    p = _lib.BrlParams(10, 0, 0, 0, 100, _lib.F_PLAYER_MODELS, 0, 2, -1.0, 1.0, 0.0, 0.0)
    assert fn(None, (ctypes.c_void_p * 6)(4096, 4096, 4096, None, None, 4096), ctypes.byref(p), ctypes.sizeof(p)) == -2
    assert b"BRL_F_PLAYER_MODELS" in L.brl_last_error()
    # brl_duplicate_match: a misaligned histogram [21]
    dup = L.brl_duplicate_match
    dup.restype, dup.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]
    fake = [4096] * 3 + [None, None, 4096, 4096, 4096, 4096] + [None] * 12 + [4098]
    p = _lib.BrlParams(100, 0, 0, 0, 100, 0, 0, 2, -1.0, 1.0, 0.0, 0.0)
    assert dup(None, (ctypes.c_void_p * 22)(*fake), ctypes.byref(p), ctypes.sizeof(p)) == -2
    assert b"[21]" in L.brl_last_error()


def test_script_parses_its_arguments():
    import importlib
    script = importlib.import_module("scripts.bidding_system")
    cfg = script.parse_args(["nets=a.pkl,b.pkl", "num_eval_envs=64", "opponent=1"])
    assert script.net_paths(cfg) == ["a.pkl", "b.pkl"] and cfg["num_eval_envs"] == 64 and cfg["opponent"] == 1
    assert script.parse_args(["data=x.txt"])["data"] == "x.txt"
    with pytest.raises(SystemExit):
        script.parse_args([])
    with pytest.raises(SystemExit):
        script.parse_args(["nope=1", "nets=a.pkl"])
