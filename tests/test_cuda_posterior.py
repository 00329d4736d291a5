"""brl_hand_posterior (DESIGN.md f18) on the GPU against tests/posterior_ref.py.

Likelihood bar: the forward tests hold each logit within BAR x the logits' range (tests/test_cuda_forward_scale.py: 5e-5 for
the default 3-term split, 2e-2 for BRL_F_MLP_BF16).  A log-softmax moves by at most twice its inputs' largest error, so log w,
a sum over the prefix's other-seat calls, is held within sum_k 2 x BAR x range_k, plus f32 rounding (1e-5 relative per
call), range_k = the largest |logit| of the float64 reference at call k.  Outputs start as 0xFF bytes (NaN)."""
import numpy as np
import pytest
import torch

from tests import helpers as H
from tests import posterior_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FORCE_LAYERS, FORCE_FUSED = 1 << 29, 1 << 30
BAR, BAR_BF16 = 5e-5, 2e-2


def _nets(seeds):
    return [H.seeded_params(s, DEV) for s in seeds]


def _np(params):
    from brl_b200.models import params_to_numpy
    return params_to_numpy(params)


def _poisoned(shape, dtype):
    t = torch.empty(shape, dtype=dtype, device=DEV)
    t.view(torch.uint8).fill_(0xFF)
    return t


def _run_op(nets, table, calls, offsets, query, seat_nets, N, *, board=None, dealer=None, vul=None, seed=0, query_offset=0,
            tau=1.0, bf16=False, path=0, capacity=None):
    """one ops.hand_posterior call with poisoned outputs -> dict of numpy arrays"""
    from brl_b200 import ops, posterior
    from brl_b200.models import ForwardPass
    pool = ops.mlp_pack_pool(nets, ForwardPass(precision="tc-bf16" if bf16 else None).pack_into)
    Q = query.shape[0]
    if capacity is None:
        dl = np.zeros(len(offsets) - 1, np.int64) if dealer is None else np.asarray(dealer, np.int64)
        segs = posterior.query_segments(query, seat_nets, dl[query[:, 0]])
        tot = {}
        for sg in segs:
            for m, n in sg.items():
                tot[m] = tot.get(m, 0) + n
        capacity = posterior._padded(tot, N)
    t = lambda a, dt: None if a is None else torch.as_tensor(np.ascontiguousarray(a, dtype=dt), device=DEV)  # noqa: E731
    out = dict(cards=_poisoned((Q, 3, 52), torch.float64), features=_poisoned((Q, 3, 95), torch.float64),
               weights=_poisoned((Q, 4), torch.float64), status=_poisoned(Q, torch.int32), hands=_poisoned((Q, N, 4), torch.int64),
               logw=_poisoned((Q, N), torch.float64))
    scratch = _poisoned(ops.hand_posterior_scratch_bytes(Q, N, capacity, len(nets)), torch.uint8)
    ops.hand_posterior(t(table, np.uint8), t(calls, np.uint8), t(offsets, np.int64), t(query, np.int32), t(seat_nets, np.int32), pool,
                       scratch, out["cards"], out["features"], out["weights"], out["status"], samples=N, row_capacity=capacity,
                       board=t(board, np.int32), dealer=t(dealer, np.int8), vul=t(vul, np.uint8), seed=seed, query_offset=query_offset,
                       temperature=tau, single_bf16=bf16, path_flags=path, hands=out["hands"], logw=out["logw"])
    torch.cuda.synchronize()
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res["hands"] = res["hands"].view(np.uint64)
    return res


def _golden(n_auctions=40):
    g = H.load_auctions()
    boards = H.load_boards()
    off = g["offsets"][:n_auctions + 1].astype(np.int64)
    calls = g["calls"][:off[-1]].astype(np.uint8)
    return boards["table"], calls, off, g


def _synthetic(n=24, seed=3):
    """auctions of random legal calls (oracle random-legal play) on a synthetic table, every dealer and vulnerability"""
    from brl_b200.deals import synthetic_deal_table
    from oracle import oracle as orc
    table = synthetic_deal_table(n, seed=seed)
    dealer = (np.arange(n) % 4).astype(np.int8)
    vul = ((np.arange(n) // 4) % 4).astype(np.uint8)
    env = orc.OracleEnv(table, n)
    env.reset_fields(np.arange(n), dealer, vul & 1, vul >> 1, np.tile(np.arange(4, dtype=np.int8), (n, 1)))
    hist = [[] for _ in range(n)]
    for step in range(40):
        ex = env.export()
        act = env.random_legal_actions(seed, step)
        for i in range(n):
            if not ex["terminated"][i]:
                hist[i].append(int(act[i]))
        env.step(act)
    off = np.cumsum([0] + [len(h) for h in hist]).astype(np.int64)
    return table, np.concatenate([np.array(h, np.uint8) for h in hist]), off, dealer, vul


def _owners_mask(table, row, seat):
    return int(np.ascontiguousarray(table[row, 8 * seat:8 * seat + 8]).view(np.uint64)[0])


# ---- sampler -----------------------------------------------------------------------------------------------------------------
def test_sampler_matches_restatement_and_partitions_the_deck():
    table, calls, off, _g = _golden(8)
    nets = _nets([1])
    query = np.array([[t, t % 4, 0] for t in range(8)], np.int32)  # L = 0: no rows, the prior
    N = 64
    res = _run_op(nets, table, calls, off, query, np.zeros((8, 4), np.int32), N, seed=11, query_offset=5)
    assert (res["status"] == 0).all()
    for j in range(8):
        s = int(query[j, 1])
        own = _owners_mask(table, j, s)
        for i in range(N):
            h = [int(x) for x in res["hands"][j, i]]
            assert h[s] == own
            assert all(bin(x).count("1") == 13 for x in h)
            assert h[0] | h[1] | h[2] | h[3] == (1 << 52) - 1
            if i < 8:
                assert h == R.sample_hands(own, s, 11, 5 + j, i), (j, i)
    # the prior: log w = 0 everywhere, W = N
    assert (res["logw"] == 0).all() and (res["weights"][:, 1] == N).all() and (res["weights"][:, 3] == N).all()


def test_sampler_is_independent_of_batching_and_chunking():
    table, calls, off, _g = _golden(6)
    nets = _nets([1])
    query = np.array([[t, (t + 1) % 4, 0] for t in range(6)], np.int32)
    whole = _run_op(nets, table, calls, off, query, np.zeros((6, 4), np.int32), 32, seed=4)
    for b, e in ((0, 2), (2, 5), (5, 6)):
        part = _run_op(nets, table, calls, off, query[b:e], np.zeros((e - b, 4), np.int32), 32, seed=4, query_offset=b)
        assert (part["hands"] == whole["hands"][b:e]).all()


def test_sampler_chi_square_card_to_seat():
    from scipy import stats
    table, calls, off, _g = _golden(4)
    nets = _nets([1])
    Q, N = 16, 65536  # 1,048,576 samples
    query = np.array([[j % 4, j % 4, 0] for j in range(Q)], np.int32)
    res = _run_op(nets, table, calls, off, query, np.zeros((Q, 4), np.int32), N, seed=2024)
    for j in range(Q):
        s = int(query[j, 1])
        hidden = R.hidden_cards(_owners_mask(table, int(query[j, 0]), s))
        counts = np.zeros((len(hidden), 3))
        for r in range(3):
            h = res["hands"][j, :, (s + 1 + r) % 4]
            for k, c in enumerate(hidden):
                counts[k, r] = int(((h >> np.uint64(c)) & np.uint64(1)).sum())
        chi2 = ((counts - N / 3) ** 2 / (N / 3)).sum()
        assert stats.chi2.sf(chi2, (len(hidden) - 1) * 2) > 1e-4, (j, chi2)


# ---- likelihood --------------------------------------------------------------------------------------------------------------
def _check_logw(res, nets_np, table, calls, off, query, seat_nets, dealer, vul, board, bar, tau=1.0, n_check=16):
    for j in range(query.shape[0]):
        t, s, L = (int(x) for x in query[j])
        if res["status"][j] != 0:
            continue
        row = t if board is None else int(board[t])
        hands = [[int(x) for x in res["hands"][j, i]] for i in range(n_check)]
        by_seat = [nets_np[int(seat_nets[j, k])] for k in range(4)]
        lg = []
        d = 0 if dealer is None else int(dealer[t])
        v = 0 if vul is None else int(vul[t])
        want = R.log_weights(by_seat, calls[off[t]:off[t + 1]], s, L, d, v, hands, tau, logits_out=lg)
        tol = sum(2 * bar * max(np.abs(x).max(), 1e-3) + 1e-5 * (1 + np.abs(x).max()) for x in lg) + 1e-9
        got = res["logw"][j, :n_check]
        assert np.allclose(got, want, rtol=0, atol=tol), (j, got, want, tol)
        assert row >= 0


@pytest.mark.parametrize("bf16,path", [(False, FORCE_LAYERS), (False, FORCE_FUSED), (True, FORCE_LAYERS), (True, FORCE_FUSED)])
def test_logw_golden_auctions(bf16, path):
    table, calls, off, g = _golden(12)
    ex = dict(board=g["board"][:12], dealer=g["dealer"][:12], vul=g["vul_ns"][:12] | (g["vul_ew"][:12] << 1))
    nets = _nets([1, 2, 3, 4])
    nets_np = [_np(p) for p in nets]
    lens = np.diff(off)
    query = np.array([[t, (t + k) % 4, int(min(lens[t], 1 + (t * 5 + k * 3) % (lens[t] + 1)))] for t in range(12) for k in range(2)],
                     np.int32)
    seat_nets = np.tile(np.array([0, 1, 2, 3], np.int32), (query.shape[0], 1))
    res = _run_op(nets, table, calls, off, query, seat_nets, 64, bf16=bf16, path=path, seed=9, **ex)
    assert (res["status"] == 0).all()
    _check_logw(res, nets_np, table, calls, off, query, seat_nets, ex["dealer"], ex["vul"], ex["board"], BAR_BF16 if bf16 else BAR)


@pytest.mark.parametrize("M", [1, 2, 4])
def test_logw_synthetic_every_dealer_vul_and_prefix(M):
    table, calls, off, dealer, vul = _synthetic()
    nets = _nets([7, 8, 9, 10][:M])
    nets_np = [_np(p) for p in nets]
    lens = np.diff(off)
    query = np.array([[t, (t * 3) % 4, L] for t in range(0, 24, 2) for L in range(0, int(lens[t]) + 1, 3)], np.int32)
    seat_nets = np.array([[(k + j) % M for k in range(4)] for j in range(query.shape[0])], np.int32)
    res = _run_op(nets, table, calls, off, query, seat_nets, 32, dealer=dealer, vul=vul, seed=5)
    assert (res["status"] == 0).all()
    _check_logw(res, nets_np, table, calls, off, query, seat_nets, dealer, vul, None, BAR, n_check=8)


def test_tau_zero_accepted_count_matches_restatement():
    table, calls, off, _g = _golden(10)
    nets = _nets([1, 2])
    nets_np = [_np(p) for p in nets]
    lens = np.diff(off)
    query = np.array([[t, t % 4, int(min(lens[t], 4))] for t in range(10)], np.int32)
    seat_nets = np.tile(np.array([0, 1, 0, 1], np.int32), (10, 1))
    N = 128
    res = _run_op(nets, table, calls, off, query, seat_nets, N, tau=0.0, seed=3)
    for j in range(10):
        t, s, L = (int(x) for x in query[j])
        hands = [[int(x) for x in res["hands"][j, i]] for i in range(N)]
        want = R.log_weights([nets_np[int(x)] for x in seat_nets[j]], calls[off[t]:off[t + 1]], s, L, 0, 0, hands, 0.0)
        assert int(res["weights"][j, 3]) == int(np.isfinite(want).sum()), j
        assert ((res["logw"][j] == 0) == np.isfinite(want)).all()


# ---- reduction ---------------------------------------------------------------------------------------------------------------
def test_reduction_matches_restatement_and_repeats_bit_for_bit():
    table, calls, off, _g = _golden(6)
    nets = _nets([1, 2])
    lens = np.diff(off)
    query = np.array([[t, (t + 2) % 4, int(lens[t])] for t in range(6)], np.int32)
    seat_nets = np.tile(np.array([0, 1, 0, 1], np.int32), (6, 1))
    a = _run_op(nets, table, calls, off, query, seat_nets, 256, seed=8)
    b = _run_op(nets, table, calls, off, query, seat_nets, 256, seed=8)
    for k in ("cards", "features", "weights", "status", "hands", "logw"):
        assert a[k].tobytes() == b[k].tobytes(), k
    for j in range(6):
        c, f, w = R.reduce(a["logw"][j], a["hands"][j], int(query[j, 1]))
        if w[3] == 0:
            assert a["weights"][j, 3] == 0 and np.isnan(a["cards"][j]).all()
            continue
        np.testing.assert_allclose(a["cards"][j], c, rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(a["features"][j], f, rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(a["weights"][j], w, rtol=1e-12)


def test_chunked_driver_is_bit_equal_to_one_chunk():
    from brl_b200 import posterior
    table, calls, off, _g = _golden(10)
    nets = _nets([1, 2])
    lens = np.diff(off)
    query = np.array([[t, s, int(lens[t])] for t in range(10) for s in range(2)], np.int32)
    seat_nets = np.tile(np.array([0, 1, 0, 1], np.int32), (20, 1))
    kw = dict(samples=64, seed=1, diagnostics=True, path_flags=FORCE_FUSED)
    one = posterior.hand_posterior(nets, table, calls, off, query, seat_nets, row_budget=1 << 20, **kw)
    many = posterior.hand_posterior(nets, table, calls, off, query, seat_nets, row_budget=2048, **kw)
    for k in ("cards", "features", "weights", "status", "hands", "logw"):
        assert one[k].tobytes() == many[k].tobytes(), k


# ---- semantics -----------------------------------------------------------------------------------------------------------------
def _blind_net(seed):
    p = H.seeded_params(seed, DEV)
    p["actor_critic/linear"]["w"][428:480] = 0  # no weight on the 52 hand bits
    return p


def test_hand_blind_net_gives_the_empirical_frequencies():
    table, calls, off, _g = _golden(4)
    nets = [_blind_net(3)]
    lens = np.diff(off)
    query = np.array([[t, 1, int(lens[t])] for t in range(4)], np.int32)
    N = 512
    res = _run_op(nets, table, calls, off, query, np.zeros((4, 4), np.int32), N, seed=6)
    for j in range(4):
        if res["status"][j]:
            continue
        assert res["weights"][j, 1] == N and res["weights"][j, 1] ** 2 / res["weights"][j, 2] == N
        s = int(query[j, 1])
        for r in range(3):
            h = res["hands"][j, :, (s + 1 + r) % 4]
            freq = np.array([((h >> np.uint64(c)) & np.uint64(1)).sum() for c in range(52)]) / N
            np.testing.assert_allclose(res["cards"][j, r], freq, rtol=1e-12, atol=1e-15)


def _analytic_net(card, call, beta):
    """a net whose only signal: hidden unit 0 = [the caller holds `card`] (observation bit 428 + card), passed through layers
    1-3 by unit 0, and a head weight beta on call `call`; every other weight zero"""
    from brl_b200.models import LAYERS
    p = H.seeded_params(1, DEV)
    for name in LAYERS:
        p[name]["w"].zero_()
        p[name]["b"].zero_()
    p[LAYERS[0]]["w"][428 + card, 0] = 1.0
    for k in (1, 2, 3):
        p[LAYERS[k]]["w"][0, 0] = 1.0
    p[LAYERS[4]]["w"][0, call] = beta
    return p


def test_analytic_bayes_posterior():
    """partner (North) opens 1C (call 3) with dealer North; the net gives call 3 the logit beta when the caller holds the ace of
    spades (card 51).  With q = P(North holds it | South's hand) = 13/39, a = e^beta / (e^beta + n_legal - 1) (holder) and
    b = 1 / n_legal (every logit 0): P(partner holds it | 1C) = q a / (q a + (1 - q) b)."""
    from brl_b200.deals import pack_deal_table, unpack_deal_table
    boards = H.load_boards()
    owners, dd = unpack_deal_table(boards["table"][:1])
    if owners[0, 51] == 2:  # the observer South must not hold the card
        owners[0] = np.where(owners[0] == 2, 9, owners[0])
        owners[0] = np.where(owners[0] == 0, 2, owners[0])
        owners[0] = np.where(owners[0] == 9, 0, owners[0])
    table = pack_deal_table(owners, dd)
    calls, off = np.array([3], np.uint8), np.array([0, 1], np.int64)
    beta = 2.0
    nets = [_analytic_net(51, 3, beta)]
    N = 65536
    query = np.array([[0, 2, 1]], np.int32)
    res = _run_op(nets, table, calls, off, query, np.zeros((1, 4), np.int32), N, seed=77)
    q, n_legal = 13 / 39, 36  # Pass + 35 bids before any bid
    a, b = np.exp(beta) / (np.exp(beta) + n_legal - 1), 1 / n_legal
    want = q * a / (q * a + (1 - q) * b)
    w = np.exp(res["logw"][0] - res["logw"][0].max())
    held = ((res["hands"][0, :, 0] >> np.uint64(51)) & np.uint64(1)).astype(bool)
    p = res["cards"][0, 1, 51]
    se = np.sqrt(np.sum(w ** 2 * (held - p) ** 2)) / w.sum()
    assert abs(p - want) < 4 * se, (p, want, se)
    c, _f, _w = R.reduce(res["logw"][0], res["hands"][0], 2)
    np.testing.assert_allclose(res["cards"][0], c, rtol=1e-12, atol=1e-15)
    zero = _run_op(nets, table, calls, off, query, np.zeros((1, 4), np.int32), 4096, seed=77, tau=0.0)
    acc = zero["logw"][0] == 0
    assert acc.any() and (((zero["hands"][0, acc, 0] >> np.uint64(51)) & np.uint64(1)) == 1).all()
    assert zero["cards"][0, 1, 51] == 1.0


# ---- edge cases ----------------------------------------------------------------------------------------------------------------
def test_edge_cases():
    from brl_b200 import _lib, ops
    table, calls, off, _g = _golden(4)
    nets = _nets([1, 2])
    lens = np.diff(off)
    # Q = 0 with NULL buffers is a no-op
    _lib.call("brl_hand_posterior", torch.cuda.current_stream().cuda_stream, [None] * 16,
              _lib.BrlParams(0, 0, 0, 0, 1, 0, 16, 1, -1.0, 1.0, 1.0, 0.0))
    bad_calls = calls.copy()
    bad_calls[off[1] + 1] = 2  # XX without a double: illegal
    query = np.array([[0, 0, int(lens[0]) + 1], [1, 0, 3], [2, 0, int(lens[2])], [3, 0, int(lens[3])]], np.int32)
    seat_nets = np.array([[0, 0, 0, 0], [0, 0, 0, 0], [0, 5, 0, 0], [0, 1, 0, 1]], np.int32)
    res = _run_op(nets, table, bad_calls, off, query, seat_nets, 16)
    assert res["status"].tolist() == [_lib.POST_SHORT, _lib.POST_ILLEGAL, _lib.POST_BAD_NET, _lib.POST_OK]
    for j in range(3):
        assert np.isnan(res["cards"][j]).all() and np.isnan(res["features"][j]).all() and res["weights"][j, 3] == 0
    assert np.isfinite(res["cards"][3]).all()
    # too small a row capacity: every query gets the capacity status
    small = _run_op(nets, table, calls, off, query[3:], seat_nets[3:], 256, capacity=256)
    assert small["status"].tolist() == [_lib.POST_CAPACITY] and np.isnan(small["cards"]).all()
    assert ops.hand_posterior_scratch_bytes(1, 256, 256, 2) > 0
