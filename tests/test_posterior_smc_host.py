"""CPU: hand reading by resample-move SMC (DESIGN.md f19) -- the float64 restatement's systematic resampling and
Metropolis-Hastings step on hand-built weights, the restated SMC against an exact Bayes posterior, the op's export, XLA
layout and argument checks (rejected before any CUDA call, through _lib.call with made-up addresses that are never
dereferenced), the host checks of ops.hand_posterior_smc and the chunk packing of method="smc"."""
import math

import numpy as np
import pytest
import torch

from brl_b200 import _lib, ops, posterior
from tests import smc_ref as S

A = 4096
OPAQUE, BUFFER = -1, -2
REQUIRED = [k for k in range(17) if k not in (3, 4, 5)]


# ---- restatement ------------------------------------------------------------------------------------------------------------
def test_systematic_resampling_on_hand_built_weights():
    w = np.array([0.0, 1.0, 0.0, 3.0])
    assert S.systematic(w, 4.0, 0.5).tolist() == [1, 3, 3, 3]  # targets 0.5, 1.5, 2.5, 3.5
    assert S.systematic(w, 4.0, 0.999).tolist() == [1, 3, 3, 3]
    assert S.systematic(np.ones(5), 5.0, 0.25).tolist() == [0, 1, 2, 3, 4]
    assert S.systematic(np.array([1.0, 0.0]), 1.0, 1 - 2 ** -40).tolist() == [0, 0]  # never past N - 1
    assert S.wants_resample(4.0, 10.0, 4, 0.5) and not S.wants_resample(4.0, 4.0, 4, 0.99) and S.wants_resample(4.0, 4.0, 4, 1.0)


def test_uniforms_and_pairs_depend_on_their_keys_only():
    u = S.resample_uniform(7, 3, 2)
    assert 0 < u < 1 and u == S.resample_uniform(7, 3, 2) != S.resample_uniform(7, 3, 3)
    assert {S.move_pair(1, g, 0, 0) for g in range(40)} == {0, 1, 2}
    a, b, lu = S.move_draws(1, 0, 0, 0, 5)
    assert 0 <= a < 13 and 0 <= b < 13 and lu < 0


def test_mh_swap_keeps_thirteen_cards_and_the_observer():
    hands = [0, 0, 0, 0]
    for c in range(52):
        hands[c // 13] |= 1 << c
    for pair in range(3):
        h = S.propose(hands, 2, pair, 0, 12)
        assert h[2] == hands[2] and all(bin(x).count("1") == 13 for x in h) and h[0] | h[1] | h[2] | h[3] == (1 << 52) - 1
        r1, r2 = S.PAIRS[pair]
        changed = [seat for seat in range(4) if h[seat] != hands[seat]]
        assert changed == sorted({(2 + 1 + r1) % 4, (2 + 1 + r2) % 4})


def _two_card_ll(beta):
    """an analytic likelihood: North (dealer) calls with weight e^beta when holding card 51, East when holding card 50"""
    def holds(h, seat, c):
        return (int(h[seat]) >> c) & 1

    def ll_n(h):
        return beta * holds(h, 0, 51) - math.log(math.exp(beta * holds(h, 0, 51)) + 35)

    def ll_e(h):
        return beta * holds(h, 1, 50) - math.log(math.exp(beta * holds(h, 1, 50)) + 35)

    def stage(k, hands):
        return np.array([ll_n(h) if k == 0 else ll_e(h) for h in hands])

    def move(k, mv, pair, hands):
        r1, r2 = S.PAIRS[pair]
        seat_ll = lambda h, seat: (ll_n(h) if seat == 0 else 0.0) + (ll_e(h) if seat == 1 and k >= 1 else 0.0)  # noqa: E731
        return np.array([[seat_ll(h, (2 + 1 + r1) % 4), seat_ll(h, (2 + 1 + r2) % 4)] for h in hands])
    return stage, move


def test_restated_smc_converges_to_the_exact_posterior():
    from tests import posterior_ref as P
    own = sum(1 << c for c in range(26, 39))  # South; both aces hidden
    beta = 2.0
    post = np.zeros((4, 4))
    for a in (0, 1, 3):
        for b in (0, 1, 3):
            prior = 13 / 39 * ((12 if a == b else 13) / 38)
            ln = math.exp(beta * (a == 0)) / (math.exp(beta * (a == 0)) + 35)
            le = math.exp(beta * (b == 1)) / (math.exp(beta * (b == 1)) + 35)
            post[a, b] = prior * ln * le
    post /= post.sum()
    stage, move = _two_card_ll(beta)
    N = 1500
    est = []
    for seed in range(4):
        hands0 = [P.sample_hands(own, 2, seed, 0, i) for i in range(N)]
        out = S.run(hands0, 2, 2, 0, seed, 0, kappa=1.0, moves=2, stage_loglik=stage, move_loglik=move)
        assert out["resamples"] == 2 and 0 < out["accepted"] < out["proposed"]
        est.append([out["cards"][1, 51], out["cards"][2, 50]])  # North is partner (1), East RHO (2)
    est = np.array(est).mean(0)
    assert abs(est[0] - post[0].sum()) < 0.05 and abs(est[1] - post[:, 1].sum()) < 0.05, (est, post[0].sum(), post[:, 1].sum())


# ---- ABI --------------------------------------------------------------------------------------------------------------------
def test_export_and_xla_layout():
    assert "brl_hand_posterior_smc" in _lib.LAZY_OPS and "brl_hand_posterior_smc_scratch_bytes" in _lib.MISC
    L = _lib.load()
    assert L.brl_xla_layout(b"brl_hand_posterior_smc") == b"iiiiiiiiisooooooo"
    assert ops.hand_posterior_smc_scratch_bytes(4, 64, 1024, 2) > ops.hand_posterior_scratch_bytes(4, 64, 1024, 2)
    assert ops.hand_posterior_smc_scratch_bytes(4, 0, 1024, 2) == -1


def _p(Q=4, *, N=64, cap=1024, M=2, tau=1.0, flags=0, n_deals=10, kappa=0.5, moves=2, stages=40, reserved=0):
    return _lib.BrlSmcParams(_lib.BrlParams(Q, 0, cap, 0, n_deals, flags, N, M, -1.0, 1.0, tau, 0.0), kappa, moves, stages, reserved)


def _bufs(drop=()):
    return [None if k in drop or k >= 17 else A * (k + 1) for k in range(25)]


def _rejects(bufs, params, code, name=None):
    with pytest.raises(_lib.BrlError) as e:
        _lib.call("brl_hand_posterior_smc", 0, bufs, params)
    assert f"({code})" in str(e.value)
    if name:
        assert f"'{name}'" in str(e.value)


def test_empty_batch_is_a_no_op():
    _lib.call("brl_hand_posterior_smc", 0, [None] * 25, _p(Q=0))


@pytest.mark.parametrize("k", REQUIRED)
def test_required_buffer(k):
    names = ["deal_table", "calls", "offsets", "board", "dealer", "vul", "query", "seat_nets", "pool", "scratch", "cards", "features",
             "weights", "status", "log_evidence", "resamples", "acceptance"]
    _rejects(_bufs(drop=(k,)), _p(), BUFFER, names[k])


@pytest.mark.parametrize("k,off", [(0, 8), (2, 4), (9, 8), (14, 4), (15, 2), (16, 4)])
def test_alignment(k, off):
    b = _bufs()
    b[k] += off
    _rejects(b, _p(), BUFFER)


def test_nullable_groups_go_together():
    b = _bufs()
    b[17], b[18] = A * 18, A * 19  # hands and logw without ell
    _rejects(b, _p(), BUFFER)
    b = _bufs()
    b[20] = A * 21  # one trace buffer of five
    _rejects(b, _p(), BUFFER)


@pytest.mark.parametrize("params", [_p(N=0), _p(M=0), _p(cap=1000), _p(tau=-0.5), _p(tau=float("nan")), _p(flags=_lib.F_SAMPLE),
                                    _p(n_deals=0), _p(kappa=-0.1), _p(kappa=1.5), _p(kappa=float("nan")), _p(moves=-1), _p(moves=65),
                                    _p(stages=-1), _p(stages=321), _p(reserved=1)])
def test_opaque_checks(params):
    _rejects(_bufs(), params, OPAQUE)


def test_short_opaque():
    with pytest.raises(_lib.BrlError, match="BrlSmcParams"):
        _lib.call("brl_hand_posterior_smc", 0, _bufs(), _lib.BrlParams(4, 0, 1024, 0, 10, 0, 64, 2, -1.0, 1.0, 1.0, 0.0))


def test_ops_wrapper_checks_before_device_work():
    table = torch.zeros((4, 48), dtype=torch.uint8)
    calls, offsets = torch.zeros(8, dtype=torch.uint8), torch.tensor([0, 4, 8], dtype=torch.int64)
    query, nets = torch.zeros((2, 3), dtype=torch.int32), torch.zeros((2, 4), dtype=torch.int32)
    f64 = lambda *s: torch.zeros(s, dtype=torch.float64)  # noqa: E731
    out = [f64(2, 3, 52), f64(2, 3, 95), f64(2, 4), torch.zeros(2, dtype=torch.int32), f64(2), torch.zeros(2, dtype=torch.int32), f64(2)]
    pool = torch.zeros((1, 16), dtype=torch.uint8)
    kw = dict(samples=16, row_capacity=256, stages=4)
    for bad, match in ((dict(moves=65), "moves"), (dict(stages=400), "stages"), (dict(ess_threshold=1.5), "ess_threshold"),
                       (dict(trace=dict(loglik=None)), "trace")):
        with pytest.raises(_lib.BrlError, match=match):
            ops.hand_posterior_smc(table, calls, offsets, query, nets, pool, None, *out, **dict(kw, **bad))
    with pytest.raises(_lib.BrlError, match="pool"):
        ops.hand_posterior_smc(table, calls, offsets, query, nets, pool, None, *out, **kw)
    with pytest.raises(_lib.BrlError, match="log_evidence"):
        ops.hand_posterior_smc(table, calls, offsets, query, nets, torch.zeros((1, ops.mlp_pool_stride()), dtype=torch.uint8), None,
                               *out[:4], f64(3), *out[5:], **kw)
    with pytest.raises(_lib.BrlError, match="go together"):
        ops.hand_posterior_smc(table, calls, offsets, query, nets, torch.zeros((1, ops.mlp_pool_stride()), dtype=torch.uint8), None,
                               *out, hands=torch.zeros((2, 16, 4), dtype=torch.int64), logw=f64(2, 16), **kw)


def test_driver_checks():
    with pytest.raises(ValueError, match="method"):
        posterior.hand_posterior([{}], None, None, [0, 1], [[0, 0, 0]], [[0, 0, 0, 0]], method="mcmc")


# ---- chunks -----------------------------------------------------------------------------------------------------------------
def test_smc_chunks_are_sized_by_the_largest_forward():
    queries = np.array([[0, 0, 8], [0, 1, 0], [0, 2, 5]], np.int32)
    nets = np.array([[0, 1, 0, 1]] * 3, np.int32)
    segs = posterior.smc_segments(queries, nets, np.zeros(3, np.int64), moves=False)
    assert segs[1] == {} and sorted(segs[0]) == [("w", k) for k in range(8) if k % 4 != 0]
    assert segs[0][("w", 1)] == {1: 1} and segs[2][("w", 4)] == {0: 1}
    # reweights only: stage k holds one call of each query whose caller at k is not its observer
    assert posterior.pack_chunks(segs, 100, 1 << 20) == [(0, 3, 256)]
    mv = posterior.smc_segments(queries, nets, np.zeros(3, np.int64), moves=True)
    # query 0 (observer North) at stage 7: East 2 calls, South 2, West 2 -> a pair holds at most 4 calls, 2 per net
    assert mv[0][("m", 7)] == {1: 4, 0: 2}
    # the largest forward is query 0's move at stage 7 (query 2 ends at stage 4): 400 + 200 rows, padded to 512 + 256
    assert posterior.pack_chunks(mv, 100, 1 << 20) == [(0, 3, 768)]
    with pytest.raises(ValueError, match="row_budget of at least"):
        posterior.pack_chunks(mv, 100, 256)
    # the IS packing is unchanged
    assert posterior.pack_chunks(posterior.query_segments(queries, nets, np.zeros(3, np.int64)), 100, 1 << 20) == [(0, 3, 512 + 768)]


def test_script_arguments():
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "scripts"))
    import hand_reading as H
    cfg = H.parse_args(["method=smc", "moves=4", "ess_threshold=0.25"])
    assert cfg["method"] == "smc" and cfg["moves"] == 4 and cfg["ess_threshold"] == 0.25
    for bad in (["method=mcmc"], ["moves=65"], ["ess_threshold=2"]):
        with pytest.raises(SystemExit):
            H.parse_args(bad)
