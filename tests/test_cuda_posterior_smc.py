"""brl_hand_posterior_smc (DESIGN.md f19) on the GPU: against brl_hand_posterior (kappa = 0 reproduces it bit for bit),
against tests/smc_ref.py fed the device's own log-likelihoods (every ancestor, pair and accept bit), and against exact Bayes
posteriors.  Outputs start as 0xFF bytes (NaN)."""
import math

import numpy as np
import pytest
import torch

from tests import helpers as H
from tests import posterior_ref as R
from tests import smc_ref as S
from tests.test_cuda_posterior import BAR, BAR_BF16, DEV, FORCE_FUSED, FORCE_LAYERS, _blind_net, _golden, _nets, _np, _poisoned, _run_op

pytestmark = pytest.mark.gpu


def _capacity(query, seat_nets, dealer, n_auctions, N, moves):
    from brl_b200 import posterior
    dl = np.zeros(n_auctions, np.int64) if dealer is None else np.asarray(dealer, np.int64)
    segs = posterior.smc_segments(query, seat_nets, dl[query[:, 0]], moves)
    return max(posterior.pack_chunks(segs, N, 1 << 30)[0][2], 256)


def _run_smc(nets, table, calls, offsets, query, seat_nets, N, *, kappa=0.5, moves=2, stages=None, board=None, dealer=None,
             vul=None, seed=0, query_offset=0, tau=1.0, bf16=False, path=0, capacity=None, trace=False):
    """one ops.hand_posterior_smc call with poisoned outputs -> dict of numpy arrays"""
    from brl_b200 import ops
    from brl_b200.models import ForwardPass
    pool = ops.mlp_pack_pool(nets, ForwardPass(precision="tc-bf16" if bf16 else None).pack_into)
    Q = query.shape[0]
    K = int(query[:, 2].max()) if stages is None else stages
    if capacity is None:
        capacity = _capacity(query, seat_nets, dealer, len(offsets) - 1, N, moves > 0 and kappa > 0)
    t = lambda a, dt: None if a is None else torch.as_tensor(np.ascontiguousarray(a, dtype=dt), device=DEV)  # noqa: E731
    out = dict(cards=_poisoned((Q, 3, 52), torch.float64), features=_poisoned((Q, 3, 95), torch.float64),
               weights=_poisoned((Q, 4), torch.float64), status=_poisoned(Q, torch.int32), log_evidence=_poisoned(Q, torch.float64),
               resamples=_poisoned(Q, torch.int32), acceptance=_poisoned(Q, torch.float64), hands=_poisoned((Q, N, 4), torch.int64),
               logw=_poisoned((Q, N), torch.float64), ell=_poisoned((Q, N, 3), torch.float64))
    tr = None
    if trace:
        tr = ops.smc_trace(Q, N, K, moves, DEV)
        for v in tr.values():
            v.view(torch.uint8).fill_(0xFF)
    scratch = _poisoned(ops.hand_posterior_smc_scratch_bytes(Q, N, capacity, len(nets)), torch.uint8)
    ops.hand_posterior_smc(t(table, np.uint8), t(calls, np.uint8), t(offsets, np.int64), t(query, np.int32), t(seat_nets, np.int32),
                           pool, scratch, out["cards"], out["features"], out["weights"], out["status"], out["log_evidence"],
                           out["resamples"], out["acceptance"], samples=N, row_capacity=capacity, stages=K, moves=moves,
                           ess_threshold=kappa, board=t(board, np.int32), dealer=t(dealer, np.int8), vul=t(vul, np.uint8), seed=seed,
                           query_offset=query_offset, temperature=tau, single_bf16=bf16, path_flags=path, hands=out["hands"],
                           logw=out["logw"], ell=out["ell"], trace=tr)
    torch.cuda.synchronize()
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res["hands"] = res["hands"].view(np.uint64)
    if trace:
        res["trace"] = {k: v.cpu().numpy() for k, v in tr.items()}
    return res


def _golden_queries(n=12, per=2):
    table, calls, off, g = _golden(n)
    ex = dict(board=g["board"][:n], dealer=g["dealer"][:n], vul=g["vul_ns"][:n] | (g["vul_ew"][:n] << 1))
    lens = np.diff(off)
    query = np.array([[t, (t + k) % 4, int(min(lens[t], 1 + (t * 5 + k * 3) % (lens[t] + 1)))] for t in range(n) for k in range(per)],
                     np.int32)
    return table, calls, off, ex, query


POST_KEYS = ("cards", "features", "weights", "status", "hands", "logw")


# ---- 1. kappa = 0 is brl_hand_posterior ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,bf16,path,tau", [(1, False, FORCE_LAYERS, 1.0), (2, False, FORCE_FUSED, 1.0), (4, True, FORCE_LAYERS, 1.0),
                                             (4, True, FORCE_FUSED, 0.5), (2, False, FORCE_LAYERS, 0.0), (4, False, FORCE_FUSED, 1.0)])
def test_kappa_zero_is_importance_sampling_bit_for_bit(M, bf16, path, tau):
    table, calls, off, ex, query = _golden_queries()
    nets = _nets([1, 2, 3, 4][:M])
    seat_nets = np.array([[(k + j) % M for k in range(4)] for j in range(query.shape[0])], np.int32)
    want = _run_op(nets, table, calls, off, query, seat_nets, 64, bf16=bf16, path=path, seed=9, tau=tau, **ex)
    got = _run_smc(nets, table, calls, off, query, seat_nets, 64, kappa=0.0, moves=3, bf16=bf16, path=path, seed=9, tau=tau, **ex)
    assert (want["status"] == 0).all()
    for k in POST_KEYS:
        assert want[k].tobytes() == got[k].tobytes(), k
    assert (got["resamples"] == 0).all() and np.isnan(got["acceptance"]).all()
    w = want["weights"]
    with np.errstate(divide="ignore"):
        ev = np.where(w[:, 3] > 0, np.log(w[:, 1] / 64) + w[:, 0], -np.inf)
    np.testing.assert_array_equal(got["log_evidence"], ev)


def test_kappa_zero_random_legal_auctions():
    from tests.test_cuda_posterior import _synthetic
    table, calls, off, dealer, vul = _synthetic()
    nets = _nets([7, 8])
    lens = np.diff(off)
    query = np.array([[t, (t * 3) % 4, L] for t in range(0, 24, 2) for L in range(0, int(lens[t]) + 1, 4)], np.int32)
    seat_nets = np.array([[(k + j) % 2 for k in range(4)] for j in range(query.shape[0])], np.int32)
    want = _run_op(nets, table, calls, off, query, seat_nets, 32, dealer=dealer, vul=vul, seed=5, path=FORCE_FUSED)
    got = _run_smc(nets, table, calls, off, query, seat_nets, 32, kappa=0.0, moves=1, dealer=dealer, vul=vul, seed=5, path=FORCE_FUSED)
    for k in POST_KEYS:
        assert want[k].tobytes() == got[k].tobytes(), k


# ---- 2. exact replay of the device's draws ------------------------------------------------------------------------------------
@pytest.mark.parametrize("kappa,tau", [(1.0, 1.0), (0.5, 1.0), (0.5, 0.0)])
def test_exact_replay_of_ancestors_and_accepts(kappa, tau):
    table, calls, off, ex, query = _golden_queries(6, 1)
    nets = _nets([1, 2])
    nets_np = [_np(p) for p in nets]
    seat_nets = np.tile(np.array([0, 1, 0, 1], np.int32), (query.shape[0], 1))
    N, moves, seed, g0 = 64, 2, 21, 3
    res = _run_smc(nets, table, calls, off, query, seat_nets, N, kappa=kappa, moves=moves, seed=seed, query_offset=g0, tau=tau,
                   path=FORCE_LAYERS, trace=True, **ex)
    tr = res["trace"]
    assert (res["status"] == 0).all()
    for j in range(query.shape[0]):
        t, s, L = (int(x) for x in query[j])
        d = int(ex["dealer"][t])
        own = int(np.ascontiguousarray(table[int(ex["board"][t]), 8 * s:8 * s + 8]).view(np.uint64)[0])
        hands0 = [S.P.sample_hands(own, s, seed, g0 + j, i) for i in range(N)]
        ref = S.run(hands0, s, L, d, seed, g0 + j, kappa=kappa, moves=moves,
                    stage_loglik=lambda k, _h: tr["loglik"][j, k],
                    move_loglik=lambda k, mv, _p, _h: tr["proposed"][j, k, mv])
        for k in range(tr["ancestors"].shape[1]):
            if k in ref["ancestors"]:
                np.testing.assert_array_equal(tr["ancestors"][j, k], ref["ancestors"][k], err_msg=f"{j} {k}")
            else:
                assert (tr["ancestors"][j, k] == -1).all(), (j, k)
            for mv in range(moves):
                if (k, mv) in ref["pairs"]:
                    assert tr["pairs"][j, k, mv] == ref["pairs"][(k, mv)]
                    np.testing.assert_array_equal(tr["accepted"][j, k, mv].astype(bool), ref["accept"][(k, mv)])
                else:
                    assert tr["pairs"][j, k, mv] == -1
        assert [[int(x) for x in h] for h in res["hands"][j]] == ref["hands"], j
        np.testing.assert_array_equal(res["logw"][j], ref["logw"])
        np.testing.assert_array_equal(res["ell"][j], ref["ell"])
        assert res["resamples"][j] == ref["resamples"]
        if ref["proposed"]:
            assert res["acceptance"][j] == ref["accepted"] / ref["proposed"]
        np.testing.assert_allclose(res["log_evidence"][j], ref["evidence"], rtol=1e-12)
        # the device's log-likelihoods against the float64 forward: the final particles' ell sums are their full log w
        if tau > 0:
            lg = []
            hands = [[int(x) for x in res["hands"][j, i]] for i in range(8)]
            want = R.log_weights([nets_np[int(x)] for x in seat_nets[j]], calls[off[t]:off[t + 1]], s, L, d,
                                 int(ex["vul"][t]), hands, tau, logits_out=lg)
            tol = sum(2 * BAR * max(np.abs(x).max(), 1e-3) + 1e-5 * (1 + np.abs(x).max()) for x in lg) + 1e-9
            np.testing.assert_allclose(res["ell"][j, :8].sum(1), want, rtol=0, atol=tol)


# ---- 3. a hand-blind net ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kappa", [0.0, 0.5, 0.99, 1.0])
def test_hand_blind_net(kappa):
    table, calls, off, _g = _golden(4)
    nets = [_blind_net(3)]
    lens = np.diff(off)
    query = np.array([[t, 1, int(lens[t])] for t in range(4)], np.int32)
    N = 256
    res = _run_smc(nets, table, calls, off, query, np.zeros((4, 4), np.int32), N, kappa=kappa, moves=2, seed=6)
    for j in range(4):
        assert res["status"][j] == 0
        assert res["weights"][j, 1] == N and res["weights"][j, 1] ** 2 / res["weights"][j, 2] == N
        if kappa < 1.0:
            assert res["resamples"][j] == 0 and np.isnan(res["acceptance"][j])
        else:
            assert res["resamples"][j] > 0 and res["acceptance"][j] == 1.0
        s = int(query[j, 1])
        for r in range(3):
            h = res["hands"][j, :, (s + 1 + r) % 4]
            freq = np.array([((h >> np.uint64(c)) & np.uint64(1)).sum() for c in range(52)]) / N
            np.testing.assert_allclose(res["cards"][j, r], freq, rtol=1e-12, atol=1e-15)


# ---- 4. a two-card analytic auction ---------------------------------------------------------------------------------------------
def _two_card_net(beta):
    """logit beta on 1C (call 3) when the caller holds the spade ace (card 51), beta on 1D (call 4) when it holds the heart
    ace (card 50), every other logit 0"""
    from brl_b200.models import LAYERS
    p = H.seeded_params(1, DEV)
    for name in LAYERS:
        p[name]["w"].zero_()
        p[name]["b"].zero_()
    p[LAYERS[0]]["w"][428 + 51, 0] = 1.0
    p[LAYERS[0]]["w"][428 + 50, 1] = 1.0
    for k in (1, 2, 3):
        p[LAYERS[k]]["w"][0, 0] = 1.0
        p[LAYERS[k]]["w"][1, 1] = 1.0
    p[LAYERS[4]]["w"][0, 3] = beta
    p[LAYERS[4]]["w"][1, 4] = beta
    return p


def _two_card_exact(beta, tau):
    """P(holder of card 51 = seat a, holder of card 50 = seat b | N 1C, E 1D) over a, b in {N, E, W}, South observing"""
    post = np.zeros((4, 4))
    for a in (0, 1, 3):
        for b in (0, 1, 3):
            prior = 13 / 39 * ((12 if a == b else 13) / 38)
            legal_n = [0] + list(range(3, 38))  # North opens: Pass and the 35 bids
            lg = np.zeros(38)
            lg[3] = beta * (a == 0)
            lg[4] = beta * (b == 0)
            lN = lg[legal_n]
            legal_e = [0, 1] + list(range(4, 38))  # East after 1C: Pass, X and the bids above 1C
            lgE = np.zeros(38)
            lgE[4] = beta * (b == 1)
            lE = lgE[legal_e]
            if tau == 0:
                like = float(legal_n[int(np.argmax(lN))] == 3) * float(legal_e[int(np.argmax(lE))] == 4)
            else:
                like = (np.exp(lg[3] / tau) / np.exp(lN / tau).sum()) * (np.exp(lgE[4] / tau) / np.exp(lE / tau).sum())
            post[a, b] = prior * like
    return post / post.sum()


@pytest.mark.parametrize("tau", [1.0, 0.0])
def test_two_card_auction_converges_to_bayes(tau):
    from brl_b200.deals import pack_deal_table
    owners = (np.arange(52) // 13).astype(np.int64)  # South holds 26..38; both aces are hidden
    table = pack_deal_table(owners[None], np.zeros((1, 4, 5), np.int64))
    calls, off = np.array([3, 4], np.uint8), np.array([0, 2], np.int64)
    beta = 2.0
    nets = [_two_card_net(beta)]
    query = np.array([[0, 2, 2]], np.int32)
    exact = _two_card_exact(beta, tau)
    rel = {1: 2, 3: 0, 0: 1}  # seat -> relative seat of South (LHO West, partner North, RHO East)
    want = {(c, seat): (exact[seat].sum() if c == 51 else exact[:, seat].sum()) for c in (50, 51) for seat in (0, 1, 3)}
    runs = [_run_smc(nets, table, calls, off, query, np.zeros((1, 4), np.int32), 4096, kappa=1.0, moves=4, seed=100 + k, tau=tau)
            for k in range(8)]
    for (c, seat), p in want.items():
        got = np.array([r["cards"][0, rel[seat], c] for r in runs])
        se = got.std(ddof=1) / math.sqrt(len(got))
        if p in (0.0, 1.0):
            assert (got == p).all(), (c, seat, got, p)
        else:
            assert abs(got.mean() - p) < 4 * max(se, 1e-4), (c, seat, got.mean(), p, se)


# ---- 5. the evidence is unbiased ------------------------------------------------------------------------------------------------
def test_evidence_agrees_with_importance_sampling():
    table, calls, off, g = _golden(8)
    ex = dict(board=g["board"][:8], dealer=g["dealer"][:8], vul=g["vul_ns"][:8] | (g["vul_ew"][:8] << 1))
    lens = np.diff(off)
    query = np.array([[t, t % 4, int(min(lens[t], 4))] for t in range(8)], np.int32)
    seat_nets = np.tile(np.array([0, 1, 0, 1], np.int32), (8, 1))
    nets = _nets([1, 2])
    smc, iss = [], []
    for k in range(16):
        a = _run_smc(nets, table, calls, off, query, seat_nets, 256, kappa=1.0, moves=2, seed=k, **ex)
        b = _run_op(nets, table, calls, off, query, seat_nets, 256, seed=1000 + k, **ex)
        smc.append(np.exp(a["log_evidence"]))
        iss.append(b["weights"][:, 1] / 256 * np.exp(b["weights"][:, 0]))
    smc, iss = np.array(smc), np.array(iss)
    for j in range(8):
        se = math.sqrt(smc[:, j].var(ddof=1) / 16 + iss[:, j].var(ddof=1) / 16)
        assert abs(smc[:, j].mean() - iss[:, j].mean()) <= 4 * se + 1e-12 * iss[:, j].mean(), (j, smc[:, j].mean(), iss[:, j].mean(), se)


# ---- 6. temperature 0 ---------------------------------------------------------------------------------------------------------
def test_tau_zero_survivors_make_every_call_and_fewer_queries_die():
    table, calls, off, g = _golden(40)
    ex = dict(board=g["board"][:40], dealer=g["dealer"][:40], vul=g["vul_ns"][:40] | (g["vul_ew"][:40] << 1))
    lens = np.diff(off)
    query = np.array([[t, s, int(lens[t])] for t in range(40) for s in range(4)], np.int32)
    seat_nets = np.tile(np.array([0, 1, 0, 1], np.int32), (query.shape[0], 1))
    nets = _nets([1, 2])
    nets_np = [_np(p) for p in nets]
    smc = _run_smc(nets, table, calls, off, query, seat_nets, 256, kappa=0.5, moves=4, tau=0.0, seed=3, **ex)
    iss = _run_op(nets, table, calls, off, query, seat_nets, 256, tau=0.0, seed=3, **ex)
    assert (smc["weights"][:, 3] == 0).mean() <= (iss["weights"][:, 3] == 0).mean()
    for j in range(0, query.shape[0], 10):
        t, s, L = (int(x) for x in query[j])
        alive = np.flatnonzero(smc["logw"][j] == 0)[:6]
        if not alive.size:
            continue
        hands = [[int(x) for x in smc["hands"][j, i]] for i in alive]
        lw = R.log_weights([nets_np[int(x)] for x in seat_nets[j]], calls[off[t]:off[t + 1]], s, L, int(ex["dealer"][t]),
                           int(ex["vul"][t]), hands, 0.0)
        assert (lw == 0).all(), j


# ---- 7. determinism, batching, edge cases ---------------------------------------------------------------------------------------
def test_bit_equal_across_repeats_chunkings_and_query_offset():
    from brl_b200 import posterior
    table, calls, off, _g = _golden(10)
    lens = np.diff(off)
    query = np.array([[t, s, int(lens[t])] for t in range(10) for s in range(2)], np.int32)
    seat_nets = np.tile(np.array([0, 1, 0, 1], np.int32), (20, 1))
    nets = _nets([1, 2])
    kw = dict(samples=64, seed=1, diagnostics=True, path_flags=FORCE_FUSED, method="smc", moves=2, ess_threshold=0.7)
    one = posterior.hand_posterior(nets, table, calls, off, query, seat_nets, row_budget=1 << 20, **kw)
    again = posterior.hand_posterior(nets, table, calls, off, query, seat_nets, row_budget=1 << 20, **kw)
    many = posterior.hand_posterior(nets, table, calls, off, query, seat_nets, row_budget=1024, **kw)
    for k in POST_KEYS + ("log_evidence", "resamples", "acceptance", "ell"):
        assert one[k].tobytes() == again[k].tobytes() == many[k].tobytes(), k
    assert one["resamples"].sum() > 0
    part = _run_smc(nets, table, calls, off, query[6:11], seat_nets[6:11], 64, kappa=0.7, moves=2, stages=int(query[:, 2].max()),
                    seed=1, query_offset=6, path=FORCE_FUSED)
    for k in POST_KEYS + ("log_evidence", "resamples", "acceptance", "ell"):
        assert part[k].tobytes() == one[k][6:11].tobytes(), k


def test_edge_cases():
    from brl_b200 import _lib, ops
    table, calls, off, _g = _golden(5)
    nets = _nets([1, 2])
    lens = np.diff(off)
    _lib.call("brl_hand_posterior_smc", torch.cuda.current_stream().cuda_stream, [None] * 25,
              _lib.BrlSmcParams(_lib.BrlParams(0, 0, 0, 0, 1, 0, 16, 1, -1.0, 1.0, 1.0, 0.0), 0.5, 1, 8, 0))
    bad_calls = calls.copy()
    bad_calls[off[1] + 1] = 2  # XX without a double: illegal
    K = int(lens[3])
    query = np.array([[0, 0, int(lens[0]) + 1], [1, 0, 3], [2, 0, int(lens[2])], [3, 0, int(lens[3])], [4, 1, int(lens[4])]], np.int32)
    seat_nets = np.array([[0, 0, 0, 0], [0, 0, 0, 0], [0, 5, 0, 0], [0, 1, 0, 1], [0, 1, 0, 1]], np.int32)
    q = query[[0, 1, 2, 3]] if lens[4] <= K else query
    res = _run_smc(nets, table, bad_calls, off, q, seat_nets[:q.shape[0]], 16, stages=K, kappa=1.0, moves=1)
    want = [_lib.POST_SHORT, _lib.POST_ILLEGAL, _lib.POST_BAD_NET, _lib.POST_OK] + ([_lib.POST_STAGES] if q.shape[0] == 5 else [])
    assert res["status"].tolist() == want
    for j in range(q.shape[0]):
        if j == 3:
            continue
        assert np.isnan(res["cards"][j]).all() and res["weights"][j, 3] == 0
        assert np.isnan(res["log_evidence"][j]) and np.isnan(res["acceptance"][j])
    assert np.isfinite(res["cards"][3]).all() and np.isfinite(res["log_evidence"][3])
    small = _run_smc(nets, table, calls, off, query[3:4], seat_nets[3:4], 256, capacity=256, kappa=1.0, moves=1)
    assert small["status"].tolist() == [_lib.POST_CAPACITY] and np.isnan(small["cards"]).all() and np.isnan(small["logw"]).all()
    assert ops.hand_posterior_smc_scratch_bytes(1, 256, 256, 2) > ops.hand_posterior_scratch_bytes(1, 256, 256, 2)
