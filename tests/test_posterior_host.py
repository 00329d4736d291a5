"""CPU: hand reading (DESIGN.md f18) -- the float64 restatement on hand-worked cases, the report statistic, the op's export,
XLA layout and argument checks (rejected before any CUDA call, through _lib.call with made-up addresses that are never
dereferenced), the host checks of ops.hand_posterior, the chunk packing and the script's argument parsing."""
import math
import os
import sys

import numpy as np
import pytest
import torch

from brl_b200 import _lib, ops, posterior
from brl_b200.deals import synthetic_deal_table, unpack_deal_table
from tests import posterior_ref as R

A = 4096
OPAQUE, BUFFER = -1, -2
NAMES = ["deal_table", "calls", "offsets", "board", "dealer", "vul", "query", "seat_nets", "pool", "scratch", "cards", "features",
         "weights", "status", "hands", "logw"]
REQUIRED = [k for k in range(14) if k not in (3, 4, 5)]


def _hand(table, row, seat):
    return int(np.ascontiguousarray(table[row, 8 * seat:8 * seat + 8]).view(np.uint64)[0])


def _const_net(bias):
    """numpy params of a net whose logits are `bias` for every observation"""
    p = {f"w{i}": np.zeros((480 if i == 0 else 1024, 1024 if i < 4 else (38 if i == 4 else 1)), np.float32) for i in range(6)}
    for i in range(6):
        p[f"b{i}"] = np.zeros(p[f"w{i}"].shape[1], np.float32)
    p["b4"] = np.asarray(bias, np.float32)
    return p


# ---- restatement ------------------------------------------------------------------------------------------------------------
def test_sampler_partitions_the_hidden_cards():
    table = synthetic_deal_table(4, seed=1)
    for s in range(4):
        own = _hand(table, s, s)
        for i in range(5):
            h = R.sample_hands(own, s, 3, 10 + s, i)
            assert h[s] == own and all(bin(x).count("1") == 13 for x in h)
            assert h[0] | h[1] | h[2] | h[3] == (1 << 52) - 1
    assert R.sample_hands(own, 3, 3, 13, 0) != R.sample_hands(own, 3, 3, 13, 1)


def test_prior_without_other_seat_calls_gives_empirical_frequencies():
    table = synthetic_deal_table(1, seed=2)
    own = _hand(table, 0, 1)
    hands = [R.sample_hands(own, 1, 0, 0, i) for i in range(40)]
    net = _const_net(np.zeros(38))
    lw = R.log_weights([net] * 4, [0], 1, 0, 0, 0, hands)  # L = 0: no call read
    assert (lw == 0).all()
    cards, feats, w = R.reduce(lw, hands, 1)
    assert w.tolist() == [0.0, 40.0, 40.0, 40.0] and R.ess(w) == 40.0
    freq = np.array([[sum((h[(1 + 1 + r) % 4] >> c) & 1 for h in hands) / 40 for c in range(52)] for r in range(3)])
    np.testing.assert_allclose(cards, freq, rtol=1e-12)
    np.testing.assert_allclose(feats.reshape(3, -1)[:, :38].sum(1), 1.0)


def test_tau_zero_accepts_exactly_the_argmax_call():
    table = synthetic_deal_table(1, seed=3)
    own = _hand(table, 0, 2)
    hands = [R.sample_hands(own, 2, 0, 0, i) for i in range(6)]
    bias = np.zeros(38)
    bias[3] = 1.0  # 1C is every net's argmax
    lw = R.log_weights([_const_net(bias)] * 4, [3], 2, 1, 0, 0, hands, tau=0.0)
    assert (lw == 0).all()
    bias[3], bias[4] = 1.0, 2.0  # 1D is, the auction shows 1C: no sample is consistent
    lw = R.log_weights([_const_net(bias)] * 4, [3], 2, 1, 0, 0, hands, tau=0.0)
    assert (lw == -np.inf).all()
    cards, feats, w = R.reduce(lw, hands, 2)
    assert np.isnan(cards).all() and np.isnan(feats).all() and np.isnan(w[:3]).all() and w[3] == 0


def test_log_softmax_over_the_legal_calls():
    table = synthetic_deal_table(1, seed=4)
    own = _hand(table, 0, 0)
    hands = [R.sample_hands(own, 0, 0, 0, 0)]
    bias = np.arange(38, dtype=np.float64) / 10
    lw = R.log_weights([_const_net(bias)] * 4, [3, 5], 0, 2, 0, 0, hands, tau=2.0)  # East's 1H after North's 1C
    legal = [0, 1] + list(range(4, 38))  # Pass, X and the bids above 1C
    x = bias[legal] / 2.0
    want = bias[5] / 2.0 - (x.max() + math.log(np.exp(x - x.max()).sum()))
    assert lw[0] == pytest.approx(want, rel=1e-6)


def test_reading_stats_on_a_hand_built_posterior():
    table = synthetic_deal_table(2, seed=5)
    owners, _ = unpack_deal_table(table)
    queries = np.array([[0, 0, 4], [1, 2, 4], [1, 3, 4]], np.int32)
    seat_nets = np.array([[0, 1, 0, 1]] * 3, np.int32)
    post = dict(cards=np.zeros((3, 3, 52)), features=np.zeros((3, 3, 95)), ess=np.array([10.0, 20.0, np.nan]),
                accepted=np.array([5, 7, 0]), status=np.zeros(3, np.int32))
    for j, (t, s, _L) in enumerate(queries[:2]):  # query 0: the truth; query 1: the prior
        for r in range(3):
            seat = (s + 1 + r) % 4
            if j == 0:
                post["cards"][j, r] = owners[t] == seat
                post["features"][j, r, R.hand_features(sum(1 << c for c in range(52) if owners[t][c] == seat))[0]] = 1
            else:
                post["cards"][j, r] = np.where(owners[t] == s, 0.0, 1 / 3)
                post["features"][j, r, 10] = 1
    rep = posterior.reading_stats(post, queries, seat_nets, owners)
    assert rep["0"]["cards_read"] == pytest.approx((39 + 13) / 2) and rep["0"]["partner_cards_read"] == pytest.approx((13 + 13 / 3) / 2)
    assert rep["0"]["hcp_abs_error"]["partner"] == pytest.approx(abs(10 - R.hand_features(
        sum(1 << c for c in range(52) if owners[1][c] == 0))[0]) / 2)
    assert rep["1"]["no_accepted_sample"] == 1 and rep["1"]["cards_read"] is None
    assert rep["0"]["cards_read_prior"] == 13.0


def test_reading_queries():
    off = np.array([0, 4, 9], np.int64)
    q, sn = posterior.reading_queries(off, np.array([[0, 1, 0, 1], [1, 0, 1, 0]]), np.array([0, 3]))
    assert q.tolist() == [[0, s, 4] for s in range(4)] + [[1, s, 5] for s in range(4)]
    q, _ = posterior.reading_queries(off, np.array([[0, 1, 0, 1], [1, 0, 1, 0]]), np.array([0, 3]), at="decisions")
    assert [tuple(x) for x in q if x[0] == 1 and x[1] == 3] == [(1, 3, 0), (1, 3, 4)]


def test_describe_lines():
    post = dict(cards=np.full((1, 3, 52), 0.25), features=np.zeros((1, 3, 95)), ess=np.array([12.5]), accepted=np.array([40]),
                status=np.zeros(1, np.int32))
    post["features"][0, :, 12] = 1.0
    post["features"][0, :, 38 + 3] = post["features"][0, :, 52 + 3] = post["features"][0, :, 66 + 3] = 1.0
    post["features"][0, :, 80 + 4] = 1.0
    lines = posterior.describe(post, 0)
    assert "ESS 12.5" in lines[0] and "HCP 12.0 (10/50/90 %: 12/12/12)" in lines[1] and "spades 4.00 (mode 4)" in lines[2]
    post["accepted"][0] = 0
    assert "no sample" in posterior.describe(post, 0)[0]


# ---- chunks ---------------------------------------------------------------------------------------------------------------
def test_chunk_packing_and_budget_error():
    segs = posterior.query_segments(np.array([[0, 0, 8], [0, 1, 0], [0, 2, 5]], np.int32), np.array([[0, 1, 0, 1]] * 3, np.int32),
                                    np.zeros(3, np.int64))
    assert segs == [{1: 4, 0: 2}, {}, {0: 2, 1: 2}]  # seats 1 and 3 play net 1, seats 0 and 2 net 0
    assert posterior.pack_chunks(segs, 100, 1 << 20) == [(0, 3, 512 + 768)]
    chunks = posterior.pack_chunks(segs, 100, 768)
    assert chunks[0][0] == 0 and chunks[-1][1] == 3 and all(rows <= 768 for _b, _e, rows in chunks)
    assert all(e > b for b, e, _ in chunks)
    with pytest.raises(ValueError, match="row_budget of at least 768"):
        posterior.pack_chunks(segs, 100, 512)


# ---- the op's export, layout and checks -----------------------------------------------------------------------------------
def test_export_and_xla_layout():
    assert "brl_hand_posterior" in _lib.LAZY_OPS and "brl_hand_posterior_scratch_bytes" in _lib.MISC
    L = _lib.load()
    assert L.brl_xla_layout(b"brl_hand_posterior") == b"iiiiiiiiisoooo"
    assert ops.hand_posterior_scratch_bytes(4, 64, 1024, 2) > 1024 * 960
    assert ops.hand_posterior_scratch_bytes(4, 0, 1024, 2) == -1


def _p(Q=4, *, N=64, cap=1024, M=2, tau=1.0, flags=0, n_deals=10):
    return _lib.BrlParams(Q, 0, cap, 0, n_deals, flags, N, M, -1.0, 1.0, tau, 0.0)


def _bufs(drop=()):
    return [None if k in drop or k >= 14 else A * (k + 1) for k in range(16)]


def _rejects(bufs, params, code, name=None):
    with pytest.raises(_lib.BrlError) as e:
        _lib.call("brl_hand_posterior", 0, bufs, params)
    assert f"({code})" in str(e.value)
    if name:
        assert f"'{name}'" in str(e.value)


def test_empty_batch_is_a_no_op():
    _lib.call("brl_hand_posterior", 0, [None] * 16, _p(Q=0))


@pytest.mark.parametrize("k", REQUIRED)
def test_required_buffer(k):
    _rejects(_bufs(drop=(k,)), _p(), BUFFER, NAMES[k])


@pytest.mark.parametrize("k,off", [(0, 8), (2, 4), (6, 2), (7, 4), (9, 8), (10, 4), (13, 2)])
def test_alignment(k, off):
    b = _bufs()
    b[k] += off
    _rejects(b, _p(), BUFFER, NAMES[k])


def test_diagnostics_go_together():
    b = _bufs()
    b[14] = A * 15
    _rejects(b, _p(), BUFFER)


@pytest.mark.parametrize("params", [_p(N=0), _p(N=(1 << 24) + 1), _p(M=0), _p(cap=1000), _p(cap=-256), _p(tau=-0.5),
                                    _p(tau=float("nan")), _p(tau=float("inf")), _p(flags=_lib.F_SAMPLE), _p(n_deals=0)])
def test_opaque_checks(params):
    _rejects(_bufs(), params, OPAQUE)


def test_short_opaque():
    with pytest.raises(_lib.BrlError):
        _lib.call("brl_hand_posterior", 0, _bufs(), _lib.BrlSlParams(4, 0.0, 0))


def test_ops_wrapper_checks_before_device_work():
    table = torch.zeros((4, 48), dtype=torch.uint8)
    calls, offsets = torch.zeros(8, dtype=torch.uint8), torch.tensor([0, 4, 8], dtype=torch.int64)
    query, nets = torch.zeros((2, 3), dtype=torch.int32), torch.zeros((2, 4), dtype=torch.int32)
    out = dict(cards=torch.zeros((2, 3, 52), dtype=torch.float64), features=torch.zeros((2, 3, 95), dtype=torch.float64),
               weights=torch.zeros((2, 4), dtype=torch.float64), status=torch.zeros(2, dtype=torch.int32))
    pool = torch.zeros((1, 16), dtype=torch.uint8)
    args = lambda **kw: dict(dict(samples=16, row_capacity=256), **kw)  # noqa: E731
    with pytest.raises(_lib.BrlError, match="pool"):
        ops.hand_posterior(table, calls, offsets, query, nets, pool, None, *out.values(), **args())
    with pytest.raises(_lib.BrlError, match="query must be"):
        ops.hand_posterior(table, calls, offsets, query[:, :2], nets, pool, None, *out.values(), **args())
    with pytest.raises(_lib.BrlError, match="offsets"):
        ops.hand_posterior(table, calls, offsets.int(), query, nets, pool, None, *out.values(), **args())


def test_posterior_driver_checks():
    with pytest.raises(ValueError, match="precision"):
        posterior.hand_posterior([{}], None, None, [0, 1], [[0, 0, 0]], [[0, 0, 0, 0]], precision="fp8")
    with pytest.raises(ValueError, match="outside"):
        posterior.hand_posterior([{}], None, None, [0, 1], [[1, 0, 0]], [[0, 0, 0, 0]])


# ---- the script -----------------------------------------------------------------------------------------------------------
def test_script_arguments():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "scripts"))
    import hand_reading as S
    cfg = S.parse_args(["boards=100", "samples=256", "temperature=0"])
    assert cfg["boards"] == 100 and cfg["samples"] == 256 and cfg["temperature"] == 0.0
    cfg = S.parse_args(["hand=AKQ2.AK32.K32.32", "auction=1C,P,1H", "dealer=N", "vul=NS", "observer=S"])
    table, calls, dealer, vul, s = S.one_hand_query(cfg)
    assert calls == [3, 0, 5] and (dealer, vul, s) == (0, 1, 2) and table.shape == (1, 48)
    with pytest.raises(SystemExit):
        S.one_hand_query(S.parse_args(["hand=AKQ.AK.K.2", "auction=1C"]))  # not 13 cards
    with pytest.raises(SystemExit):
        S.parse_args(["nonsense=1"])
    with pytest.raises(SystemExit):
        S.parse_args(["auction=1C"])  # --auction without --hand
