"""Hand reading (DESIGN.md f18) in plain Python and float64: the one reference for brl_hand_posterior.  Restates the
definitions of include/brl_b200.h:

  sample i of query j (global index g): the 39 cards outside the observer's hand, in increasing card index h[0..38], are
    shuffled by Fisher-Yates, for t = 0..37 with n = 38 - t: swap h[n], h[mulhi(u_t, n + 1)], u_t = word t % 4 of
    philox4x32((g_lo, g_hi, POST_TAG + t // 4, i), (seed_lo, seed_hi)); h[0..12] -> LHO (s + 1), h[13..25] -> partner
    (s + 2), h[26..38] -> RHO (s + 3)
  log w = sum over calls k < L by a seat other than s of log softmax over the legal calls of logits / tau at c_k (tau = 0:
    0 at the masked first argmax, -inf elsewhere); the observation of caller sigma_k after c_0 .. c_{k-1} with sigma_k's
    sampled hand, built by the oracle env (OracleEnv.reset_fields / step / observe) on a deal row with the sampled owners
  posterior: M = max log w, w' = exp(log w - M), W = sum w'; cards / features are w'-weighted means; weights = {M, W, sum w'^2,
    #(w > 0)}; NaN (count 0) when no sample is accepted."""
import numpy as np

from brl_b200.deals import pack_deal_table
from oracle import oracle as orc

POST_TAG = 0x484E4430
FEATURES = 95
M32 = 0xFFFFFFFF


def hidden_cards(own_mask: int):
    return [c for c in range(52) if not (int(own_mask) >> c) & 1]


def sample_hands(own_mask: int, s: int, seed: int, g: int, i: int):
    """u64 hand masks [4] by absolute seat of sample i of the query with global index g"""
    h = hidden_cards(own_mask)
    assert len(h) == 39
    key = [seed & M32, (seed >> 32) & M32]
    u = []
    for b in range(10):
        u.extend(int(x) for x in orc.philox([g & M32, (g >> 32) & M32, POST_TAG + b, i], key))
    for t in range(38):
        n = 38 - t
        j = (u[t] * (n + 1)) >> 32
        h[n], h[j] = h[j], h[n]
    hands = [0, 0, 0, 0]
    hands[s] = int(own_mask)
    for r in range(3):
        hands[(s + 1 + r) % 4] = sum(1 << c for c in h[13 * r:13 * r + 13])
    return hands


def owners_of(hands):
    """owners[52] (seat of every card) of four u64 hand masks"""
    own = np.full(52, -1, np.int64)
    for seat in range(4):
        for c in range(52):
            if (int(hands[seat]) >> c) & 1:
                own[c] = seat
    assert (own >= 0).all()
    return own


def forward64(params_np, x):
    """logits of the DeepMind MLP in float64 (params_np: models.params_to_numpy)"""
    h = np.asarray(x, dtype=np.float64)
    for i in range(4):
        h = np.maximum(h @ params_np[f"w{i}"].astype(np.float64) + params_np[f"b{i}"].astype(np.float64), 0.0)
    return h @ params_np["w4"].astype(np.float64) + params_np["b4"].astype(np.float64)


def auction_rows(calls, s: int, L: int, dealer: int, vul: int, hands_list):
    """Replay calls[:L] on one oracle env per sample (deal rows with the sampled owners) and return, for every k < L whose
    caller is not s, (k, caller, obs u8[n, 480], legal u8[n, 38], call)."""
    n = len(hands_list)
    owners = np.stack([owners_of(h) for h in hands_list])
    table = pack_deal_table(owners, np.zeros((n, 4, 5), np.int64))
    env = orc.OracleEnv(table, n)
    env.reset_fields(np.arange(n), np.full(n, dealer), np.full(n, vul & 1), np.full(n, vul >> 1),
                     np.tile(np.arange(4, dtype=np.int8), (n, 1)))
    out = []
    for k in range(L):
        caller = (dealer + k) % 4
        c = int(calls[k])
        if caller != s:
            obs = env.observe(np.full(n, caller))
            legal = env.export()["legal_action_mask"]
            out.append((k, caller, obs, legal, c))
        env.step(np.full(n, c, np.int32))
    return out


def log_weights(params_np_by_seat, calls, s: int, L: int, dealer: int, vul: int, hands_list, tau: float = 1.0,
                logits_out=None):
    """log w f64[n] of the samples (hands_list[i] = four hand masks by absolute seat); params_np_by_seat[seat] = that seat's
    net (models.params_to_numpy).  logits_out, if a list, receives the float64 logits of every (k, sample)."""
    n = len(hands_list)
    lw = np.zeros(n, np.float64)
    for k, caller, obs, legal, c in auction_rows(calls, s, L, dealer, vul, hands_list):
        lg = forward64(params_np_by_seat[caller], obs)
        if logits_out is not None:
            logits_out.append(lg)
        leg = legal.astype(bool)
        if tau == 0.0:
            ml = np.where(leg, lg, -np.inf)
            lw += np.where(ml.argmax(1) == c, 0.0, -np.inf)
        else:
            x = np.where(leg, lg / tau, -np.inf)
            mx = x.max(1)
            lse = mx + np.log(np.exp(x - mx[:, None]).sum(1))
            lw += x[:, c] - lse
    return lw


def hand_features(mask: int):
    """(hcp, [len clubs..spades], balanced) of a u64 hand mask (card c = rank * 4 + suit)"""
    cards = [c for c in range(52) if (int(mask) >> c) & 1]
    hcp = sum(max(0, c // 4 - 8) for c in cards)
    lens = [sum(1 for c in cards if c % 4 == u) for u in range(4)]
    balanced = min(lens) >= 2 and sum(1 for x in lens if x == 2) <= 1
    return hcp, lens, balanced


def feature_row(mask: int):
    """the 95 feature columns (0 / 1) of one hand: HCP 0..37, 38 + 14 suit + length, 94 balanced"""
    row = np.zeros(FEATURES, np.float64)
    hcp, lens, bal = hand_features(mask)
    row[hcp] = 1
    for u in range(4):
        row[38 + 14 * u + lens[u]] = 1
    row[94] = float(bal)
    return row


def reduce(logw, hands, s: int):
    """(cards f64[3, 52], features f64[3, 95], weights f64[4]) of one query from its samples' log w and hands [N, 4]"""
    logw = np.asarray(logw, np.float64)
    nan = float("nan")
    mx = logw.max() if logw.size else -np.inf
    if not np.isfinite(mx):
        return np.full((3, 52), nan), np.full((3, FEATURES), nan), np.array([nan, nan, nan, 0.0])
    w = np.exp(logw - mx)
    W = 0.0
    W2 = 0.0
    for x in w:  # in sample order, as the device sums
        W += x
        W2 += x * x
    cards = np.zeros((3, 52))
    feats = np.zeros((3, FEATURES))
    for i, x in enumerate(w):
        if x == 0.0:
            continue
        for r in range(3):
            h = int(hands[i][(s + 1 + r) % 4])
            cards[r] += x * np.array([(h >> c) & 1 for c in range(52)], np.float64)
            feats[r] += x * feature_row(h)
    return cards / W, feats / W, np.array([mx, W, W2, float((w > 0).sum())])


def ess(weights):
    """effective sample size W^2 / sum w'^2 of a weights row"""
    return weights[1] ** 2 / weights[2]
