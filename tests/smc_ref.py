"""Hand reading by resample-move SMC (DESIGN.md f19) in plain Python and float64: the one reference for brl_hand_posterior_smc.
Restates the definitions of include/brl_b200.h:

  particles start as posterior_ref.sample_hands; per particle log w = 0 and ell[3] = 0 (LHO, partner, RHO)
  stage k (k < L, caller sigma != s, query not extinct): log w += l_k, ell[sigma] += l_k; M = max log w (-inf: extinct);
    w' = exp(log w - M), W, S summed in particle order; resample when kappa >= 1 or W * W / S < kappa N: u = (x + 0.5) 2^-32,
    x = philox((g_lo, g_hi, SMC_TAG + 128 k, 0xFFFFFFFF)).x; C_m = C_{m-1} + w'_m; ancestor of i = first m with
    C_m >= (i + u) W / N (at most N - 1); evidence += log(W / N) + M; log w = 0
  move mv after a resample: P(c3) = philox((g_lo, g_hi, SMC_TAG + 128 k + 1 + mv, c3)); pair = mulhi(P(0xFFFFFFFF).x, 3);
    particle i swaps card mulhi(P(i).x, 13) of r1 with card mulhi(P(i).y, 13) of r2; accepted iff
    log((P(i).z + 0.5) 2^-32) < ell'[r1] + ell'[r2] - ell[r1] - ell[r2]
  end: posterior_ref.reduce; evidence += log(W / N) + M (-inf when nothing is accepted)

The likelihood is a callback, so the same code runs an analytic likelihood or the device's own log-likelihoods read back
from the op's trace (exact replay)."""
import math

import numpy as np

from oracle import oracle as orc
from tests import posterior_ref as P

SMC_TAG = 0x534D0000
M32 = 0xFFFFFFFF
PAIRS = ((0, 1), (0, 2), (1, 2))


def _philox(g: int, word2: int, c3: int, seed: int):
    return [int(x) for x in orc.philox([g & M32, (g >> 32) & M32, word2 & M32, c3 & M32], [seed & M32, (seed >> 32) & M32])]


def resample_uniform(seed: int, g: int, k: int) -> float:
    return (_philox(g, SMC_TAG + 128 * k, M32, seed)[0] + 0.5) * 2.0 ** -32


def move_pair(seed: int, g: int, k: int, mv: int) -> int:
    return (_philox(g, SMC_TAG + 128 * k + 1 + mv, M32, seed)[0] * 3) >> 32


def move_draws(seed: int, g: int, k: int, mv: int, i: int):
    """(card index a of r1, card index b of r2, log u) of particle i"""
    x, y, z, _ = _philox(g, SMC_TAG + 128 * k + 1 + mv, i, seed)
    return (x * 13) >> 32, (y * 13) >> 32, math.log((z + 0.5) * 2.0 ** -32)


def ess_weights(logw):
    """(M, w', W, S) in particle order; M = -inf when every weight is 0"""
    logw = np.asarray(logw, np.float64)
    mx = float(logw.max())
    if mx == -math.inf:
        return mx, None, 0.0, 0.0
    w = np.exp(logw - mx)
    W = S = 0.0
    for x in w:
        W += x
        S += x * x
    return mx, w, W, S


def wants_resample(W: float, S: float, N: int, kappa: float) -> bool:
    kappa = float(np.float32(kappa))
    return kappa >= 1.0 or W * W / S < kappa * N


def systematic(w, W: float, u: float):
    """ancestors [N] of systematic resampling: the first m whose running sum C_m >= (i + u) W / N"""
    N = len(w)
    anc = np.zeros(N, np.int64)
    m, C = 0, float(w[0])
    for i in range(N):
        target = (i + u) * W / N
        while C < target and m < N - 1:
            m += 1
            C += float(w[m])
        anc[i] = m
    return anc


def nth_card(mask: int, n: int) -> int:
    return [c for c in range(52) if (int(mask) >> c) & 1][n]


def propose(hands, s: int, pair: int, a: int, b: int):
    r1, r2 = PAIRS[pair]
    s1, s2 = (s + 1 + r1) % 4, (s + 1 + r2) % 4
    h = [int(x) for x in hands]
    c1, c2 = nth_card(h[s1], a), nth_card(h[s2], b)
    h[s1] ^= (1 << c1) | (1 << c2)
    h[s2] ^= (1 << c1) | (1 << c2)
    return h


def run(hands0, s: int, L: int, dealer: int, seed: int, g: int, *, kappa: float, moves: int, stage_loglik, move_loglik,
        stages=None):
    """The SMC of one query.  hands0: N particles' four hand masks; stage_loglik(k, hands_list) -> l_k f64[N];
    move_loglik(k, mv, pair, proposed_hands_list) -> ell' f64[N, 2] (the pair's two seats, calls <= k).
    -> dict(hands, logw, ell, evidence, resamples, accepted, proposed, ancestors {k: [N]}, pairs {(k, mv): pair},
    accept {(k, mv): bool[N]})"""
    N = len(hands0)
    hands = [list(map(int, h)) for h in hands0]
    logw = np.zeros(N)
    ell = np.zeros((N, 3))
    out = dict(evidence=0.0, resamples=0, accepted=0, proposed=0, ancestors={}, pairs={}, accept={})
    live = True
    for k in range(L if stages is None else min(L, stages)):
        caller = (dealer + k) % 4
        if caller == s or not live:
            continue
        r = (caller - s - 1) % 4
        lk = np.asarray(stage_loglik(k, hands), np.float64)
        logw = logw + lk
        ell[:, r] += lk
        mx, w, W, S = ess_weights(logw)
        if mx == -math.inf:
            live = False
            continue
        if not wants_resample(W, S, N, kappa):
            continue
        anc = systematic(w, W, resample_uniform(seed, g, k))
        out["ancestors"][k] = anc
        hands = [list(hands[m]) for m in anc]
        ell = ell[anc].copy()
        logw = np.zeros(N)
        out["evidence"] += math.log(W / N) + mx
        out["resamples"] += 1
        for mv in range(moves):
            pair = move_pair(seed, g, k, mv)
            out["pairs"][(k, mv)] = pair
            r1, r2 = PAIRS[pair]
            draws = [move_draws(seed, g, k, mv, i) for i in range(N)]
            prop = [propose(hands[i], s, pair, draws[i][0], draws[i][1]) for i in range(N)]
            lp = np.asarray(move_loglik(k, mv, pair, prop), np.float64).reshape(N, 2)
            acc = np.zeros(N, bool)
            for i in range(N):
                delta = (lp[i, 0] + lp[i, 1]) - (ell[i, r1] + ell[i, r2])
                acc[i] = draws[i][2] < delta
                if acc[i]:
                    hands[i] = prop[i]
                    ell[i, r1], ell[i, r2] = lp[i, 0], lp[i, 1]
            out["accept"][(k, mv)] = acc
            out["accepted"] += int(acc.sum())
            out["proposed"] += N
    out.update(hands=hands, logw=logw, ell=ell)
    cards, feats, wt = P.reduce(logw, hands, s)
    out.update(cards=cards, features=feats, weights=wt)
    out["evidence"] = -math.inf if wt[3] == 0 else out["evidence"] + math.log(wt[1] / N) + wt[0]
    return out

