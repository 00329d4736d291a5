"""Hand reading (DESIGN.md f18): what an auction tells each seat about the three hands it cannot see, under the nets' own
policies, and how much hand information a net's auctions carry.

`hand_posterior` runs brl_hand_posterior: for each query (auction, observer seat, prefix length) it deals the 39 unseen cards
at random N times, weights every deal by the probability that the nets would have made the other seats' calls with those
hands, and returns the weighted card holdings and hand features.  With method="smc" it runs brl_hand_posterior_smc instead
(DESIGN.md f19): the same deals are reweighted call by call, resampled when their effective sample size falls below
ess_threshold x N, and moved by Metropolis-Hastings card swaps, so long auctions keep usable samples.  `describe` prints one query's posterior, and `hand_reading`
scores the posteriors of auctions whose deals are known."""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib, ops
from .deals import unpack_deal_table
from .models import ForwardPass

SEAT_NAMES = "NESW"
REL_NAMES = ("LHO", "partner", "RHO")
SUIT_NAMES = ("clubs", "diamonds", "hearts", "spades")
DEFAULT_ROW_BUDGET = 1 << 20  # forward rows per device call: about 10 KB of scratch each (obs, gather, activations, logits)


def _calls_by(seat: int, dealer: int, L: int) -> int:
    r = (seat - dealer) % 4
    return (L - 1 - r) // 4 + 1 if L > r else 0


def query_segments(queries: np.ndarray, seat_nets: np.ndarray, dealers: np.ndarray) -> List[Dict[int, int]]:
    """per query: {net: the calls of the prefix made by other seats playing that net}; a query's rows are N times their sum"""
    out = []
    for (t, s, L), nets, d in zip(queries, seat_nets, dealers):
        seg: Dict[int, int] = {}
        if 0 <= s < 4 and L > 0:
            for seat in range(4):
                n = _calls_by(seat, int(d), int(L)) if seat != s else 0
                if n:
                    seg[int(nets[seat])] = seg.get(int(nets[seat]), 0) + n
        out.append(seg)
    return out


def smc_segments(queries: np.ndarray, seat_nets: np.ndarray, dealers: np.ndarray, moves: bool) -> List[Dict]:
    """per query of brl_hand_posterior_smc: {forward: {net: calls}} over the forwards it takes part in, ("w", k) for stage k's
    reweight and, with moves, ("m", k) for the moves after a resample at stage k, at the most rows any pair of hidden seats
    can need; a chunk's forward capacity is the largest of these forwards summed over its queries"""
    out = []
    for (t, s, L), nets, d in zip(queries, seat_nets, dealers):
        seg: Dict = {}
        by_seat = [0, 0, 0, 0]
        if 0 <= s < 4:
            for k in range(int(L)):
                caller = (int(d) + k) % 4
                if caller == s:
                    continue
                by_seat[caller] += 1
                seg[("w", k)] = {int(nets[caller]): 1}
                if moves:
                    bound: Dict[int, int] = {}
                    hidden = [(int(s) + 1 + r) % 4 for r in range(3)]
                    for a, b in ((0, 1), (0, 2), (1, 2)):
                        pair: Dict[int, int] = {}
                        for seat in (hidden[a], hidden[b]):
                            if by_seat[seat]:
                                pair[int(nets[seat])] = pair.get(int(nets[seat]), 0) + by_seat[seat]
                        for m, n in pair.items():
                            bound[m] = max(bound.get(m, 0), n)
                    seg[("m", k)] = bound
        out.append(seg)
    return out


def _padded(per_net: Dict[int, int], N: int) -> int:
    return sum((N * n + 255) // 256 * 256 for n in per_net.values())


def pack_chunks(segments: Sequence[Dict], N: int, row_budget: int):
    """Consecutive query ranges [(begin, end, padded rows)] whose forward fits `row_budget` rows; a query that does not fit
    alone raises ValueError with the budget it needs.  segments[j] is query_segments' {net: calls} (one forward), or
    smc_segments' {forward: {net: calls}}: then the rows of a chunk are those of its largest forward, not their sum."""
    def rows(acc):
        return max((_padded(v, N) for v in acc.values()), default=0)

    def add(acc, seg):
        out = {key: dict(v) for key, v in acc.items()}
        for key, per_net in seg.items():
            tot = out.setdefault(key, {})
            for m, n in per_net.items():
                tot[m] = tot.get(m, 0) + n
        return out

    staged = [seg if seg and isinstance(next(iter(seg.values())), dict) else {0: seg} for seg in segments]
    chunks, begin, acc = [], 0, {}
    for j, seg in enumerate(staged):
        alone = rows(seg)
        if alone > row_budget:
            calls = max((sum(v.values()) for v in seg.values()), default=0)
            raise ValueError(f"hand_posterior: query {j} needs a row_budget of at least {alone} rows ({N} samples x "
                             f"{calls} calls by other seats), the budget is {row_budget}")
        trial = add(acc, seg)
        if j > begin and rows(trial) > row_budget:
            chunks.append((begin, j, rows(acc)))
            begin, trial = j, add({}, seg)
        acc = trial
    if begin < len(staged):
        chunks.append((begin, len(staged), rows(acc)))
    return chunks


def hand_posterior(params_list, table, calls, offsets, queries, seat_nets, *, board=None, dealer=None, vul=None, samples: int = 1024,
                   seed: int = 0, temperature: float = 1.0, precision: Optional[str] = None, row_budget: int = DEFAULT_ROW_BUDGET,
                   diagnostics: bool = False, path_flags: int = 0, method: str = "is", moves: int = 1, ess_threshold: float = 0.5,
                   device="cuda") -> Dict[str, np.ndarray]:
    """Posterior of the hidden hands for every query (t, s, L) of `queries` (int [Q, 3]): auction t of calls / offsets (u8 /
    int64, brl_sl_examples' encoding) read by absolute seat s after its first L calls, seat k playing net seat_nets[j, k] of
    params_list.  board / dealer / vul as ops.hand_posterior (None: row t, North, nobody vulnerable).  Queries are packed into
    device calls of at most `row_budget` forward rows; sample i of query j depends on (seed, j, i) only.
    -> numpy: cards [Q, 3, 52] and features [Q, 3, 95] (relative seats LHO, partner, RHO), ess [Q], accepted [Q] (samples with
    weight > 0), log_max [Q], weights [Q, 4], status [Q] (BRL_POST_*), and with diagnostics hands [Q, N, 4] (u64 masks by absolute
    seat) and logw [Q, N].
    method="smc" runs the resample-move sequential Monte Carlo sampler (ops.hand_posterior_smc) with `moves` Metropolis-Hastings
    moves after each resample and resampling when the ESS falls below ess_threshold x N; the result gains log_evidence [Q],
    resamples [Q] and acceptance [Q] (and ell [Q, N, 3] with diagnostics).  Chunks are then sized by the largest forward of
    any stage or move."""
    if precision not in (None, "tc", "tc-bf16"):
        raise ValueError(f"unknown precision {precision!r}")
    if method not in ("is", "smc"):
        raise ValueError(f"unknown method {method!r}: 'is' or 'smc'")
    smc = method == "smc"
    if not params_list:
        raise ValueError("hand_posterior: no nets")
    queries = np.ascontiguousarray(queries, dtype=np.int32).reshape(-1, 3)
    seat_nets = np.ascontiguousarray(seat_nets, dtype=np.int32).reshape(-1, 4)
    if seat_nets.shape[0] != queries.shape[0]:
        raise ValueError("hand_posterior: one row of seat_nets per query")
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    n_auctions = offsets.shape[0] - 1
    if queries.size and (queries[:, 0].min() < 0 or queries[:, 0].max() >= n_auctions):
        raise ValueError(f"hand_posterior: a query's auction is outside [0, {n_auctions})")
    N, Q = int(samples), queries.shape[0]
    dealers = np.zeros(n_auctions, np.int64) if dealer is None else np.asarray(dealer, np.int64)
    qd = dealers[queries[:, 0]] if Q else np.zeros(0, np.int64)
    segments = (smc_segments(queries, seat_nets, qd, moves > 0 and ess_threshold > 0) if smc
                else query_segments(queries, seat_nets, qd))
    chunks = pack_chunks(segments, N, row_budget)
    dev = torch.device(device)

    def t(a, dt):
        return None if a is None else torch.as_tensor(np.ascontiguousarray(a, dtype=dt), device=dev)

    table_t, calls_t, offsets_t = t(table, np.uint8), t(calls, np.uint8), t(offsets, np.int64)
    board_t, dealer_t, vul_t = t(board, np.int32), t(dealer, np.int8), t(vul, np.uint8)
    pool = ops.mlp_pack_pool(list(params_list), ForwardPass(precision=precision).pack_into)
    out = dict(cards=np.full((Q, 3, 52), np.nan), features=np.full((Q, 3, _lib.POST_FEATURES), np.nan), weights=np.zeros((Q, 4)),
               status=np.zeros(Q, np.int32))
    if diagnostics:
        out["hands"], out["logw"] = np.zeros((Q, N, 4), np.uint64), np.zeros((Q, N))
    if smc:
        out.update(log_evidence=np.full(Q, np.nan), resamples=np.zeros(Q, np.int32), acceptance=np.full(Q, np.nan))
        if diagnostics:
            out["ell"] = np.zeros((Q, N, 3))
    for b, e, rows in chunks:
        q = e - b
        size = (ops.hand_posterior_smc_scratch_bytes if smc else ops.hand_posterior_scratch_bytes)(q, N, rows, pool.shape[0])
        scratch = torch.empty(size, dtype=torch.uint8, device=dev)
        res = dict(cards=torch.empty((q, 3, 52), dtype=torch.float64, device=dev),
                   features=torch.empty((q, 3, _lib.POST_FEATURES), dtype=torch.float64, device=dev),
                   weights=torch.empty((q, 4), dtype=torch.float64, device=dev), status=torch.empty(q, dtype=torch.int32, device=dev))
        diag = {}
        if diagnostics:
            diag = dict(hands=torch.empty((q, N, 4), dtype=torch.int64, device=dev), logw=torch.empty((q, N), dtype=torch.float64, device=dev))
        args = (table_t, calls_t, offsets_t, t(queries[b:e], np.int32), t(seat_nets[b:e], np.int32), pool, scratch, res["cards"],
                res["features"], res["weights"], res["status"])
        kw = dict(samples=N, row_capacity=rows, board=board_t, dealer=dealer_t, vul=vul_t, seed=seed, query_offset=b,
                  temperature=temperature, single_bf16=precision == "tc-bf16", path_flags=path_flags, **diag)
        if smc:
            res.update(log_evidence=torch.empty(q, dtype=torch.float64, device=dev), resamples=torch.empty(q, dtype=torch.int32, device=dev),
                       acceptance=torch.empty(q, dtype=torch.float64, device=dev))
            if diagnostics:
                diag["ell"] = kw["ell"] = torch.empty((q, N, 3), dtype=torch.float64, device=dev)
            ops.hand_posterior_smc(*args, res["log_evidence"], res["resamples"], res["acceptance"],
                                   stages=int(queries[b:e, 2].max(initial=0)), moves=moves, ess_threshold=ess_threshold, **kw)
        else:
            ops.hand_posterior(*args, **kw)
        for k, v in res.items():
            out[k][b:e] = v.cpu().numpy()
        for k, v in diag.items():
            out[k][b:e] = v.cpu().numpy().view(np.uint64) if k == "hands" else v.cpu().numpy()
    w = out["weights"]
    with np.errstate(invalid="ignore", divide="ignore"):
        out["ess"] = w[:, 1] ** 2 / w[:, 2]
    out["accepted"] = w[:, 3].astype(np.int64)
    out["log_max"] = w[:, 0]
    return out


def _quantile(dist: np.ndarray, q: float) -> int:
    return int(np.searchsorted(np.cumsum(dist), q - 1e-12))


def describe(post: Dict[str, np.ndarray], j: int) -> List[str]:
    """readable lines of query j's posterior: per hidden seat the expected HCP with its 10/50/90 % points, the mean and modal
    suit lengths, P(balanced) and the probabilities of the aces and kings"""
    if post["accepted"][j] == 0:
        return [f"query {j}: no sample consistent with the auction (status {int(post['status'][j])})"]
    lines = [f"query {j}: {int(post['accepted'][j])} samples accepted, ESS {post['ess'][j]:.1f}"]
    for r, name in enumerate(REL_NAMES):
        f, c = post["features"][j, r], post["cards"][j, r]
        hcp = f[:38]
        lines.append(f"  {name}: HCP {float(np.arange(38) @ hcp):.1f} (10/50/90 %: {_quantile(hcp, .1)}/{_quantile(hcp, .5)}/"
                     f"{_quantile(hcp, .9)}), balanced {f[94]:.2f}")
        lens = [f[38 + 14 * u:52 + 14 * u] for u in range(4)]
        lines.append("    lengths " + ", ".join(f"{SUIT_NAMES[u]} {float(np.arange(14) @ lens[u]):.2f} (mode {int(lens[u].argmax())})"
                                                for u in range(4)))
        lines.append("    aces " + " ".join(f"{'CDHS'[u]}A {c[48 + u]:.2f}" for u in range(4)) +
                     "   kings " + " ".join(f"{'CDHS'[u]}K {c[44 + u]:.2f}" for u in range(4)))
    return lines


def _hcp(owners_row: np.ndarray, seat: int) -> int:
    return int(sum(max(0, c // 4 - 8) for c in range(52) if owners_row[c] == seat))


def reading_queries(offsets, seat_nets_by_auction, dealer=None, at: str = "end"):
    """(queries [Q, 3], seat_nets [Q, 4]): every auction read by each of the four seats, at its end or, with
    at="decisions", before each of that seat's own calls"""
    if at not in ("end", "decisions"):
        raise ValueError("at must be 'end' or 'decisions'")
    offsets = np.asarray(offsets, np.int64)
    nets = np.asarray(seat_nets_by_auction, np.int32).reshape(-1, 4)
    q, sn = [], []
    for t in range(offsets.shape[0] - 1):
        length = int(offsets[t + 1] - offsets[t])
        d = 0 if dealer is None else int(dealer[t])
        for s in range(4):
            prefixes = [length] if at == "end" else [k for k in range(length) if (d + k) % 4 == s]
            for L in prefixes:
                q.append((t, s, L))
                sn.append(nets[t])
    return np.array(q, np.int32).reshape(-1, 3), np.array(sn, np.int32).reshape(-1, 4)


def reading_stats(post: Dict[str, np.ndarray], queries: np.ndarray, seat_nets: np.ndarray, owners: np.ndarray,
                  board=None) -> Dict[str, Dict]:
    """The information statistic per observer net over queries with known deals (owners [rows, 52], the deal table's):
    cards read = sum over the 39 hidden cards of P(true holder) (13 under the prior), partner cards read = the same over
    partner's 13 cards (13/3 under the prior), the mean |E[HCP] - true HCP| per hidden seat, ESS quantiles and the share of
    queries without an accepted sample (excluded from the rest).  Linear in the posterior: no log of a zero probability."""
    per: Dict[int, Dict[str, list]] = {}
    for j, (t, s, _L) in enumerate(queries):
        net = int(seat_nets[j, s])
        acc = per.setdefault(net, dict(cards=[], partner=[], hcp_err=[], ess=[], empty=0, n=0))
        acc["n"] += 1
        if post["accepted"][j] == 0:
            acc["empty"] += 1
            continue
        row = owners[int(t) if board is None else int(board[t])]
        rel = (row.astype(np.int64) - int(s) - 1) % 4  # 0 LHO, 1 partner, 2 RHO, 3 the observer
        hidden = rel < 3
        p_true = post["cards"][j][rel[hidden], np.arange(52)[hidden]]
        acc["cards"].append(float(p_true.sum()))
        acc["partner"].append(float(p_true[rel[hidden] == 1].sum()))
        acc["hcp_err"].append([abs(float(np.arange(38) @ post["features"][j, r, :38]) - _hcp(row, (int(s) + 1 + r) % 4))
                               for r in range(3)])
        acc["ess"].append(float(post["ess"][j]))
    report = {}
    for net, a in sorted(per.items()):
        ok = len(a["cards"])
        err = np.array(a["hcp_err"]).reshape(-1, 3)
        report[str(net)] = dict(
            queries=a["n"], no_accepted_sample=a["empty"], no_accepted_share=a["empty"] / max(a["n"], 1),
            cards_read=float(np.mean(a["cards"])) if ok else None, cards_read_prior=13.0,
            partner_cards_read=float(np.mean(a["partner"])) if ok else None, partner_cards_read_prior=13.0 / 3.0,
            hcp_abs_error={name: (float(err[:, r].mean()) if ok else None) for r, name in enumerate(REL_NAMES)},
            ess_quantiles={f"p{q}": (float(np.percentile(a["ess"], q)) if ok else None) for q in (10, 50, 90)})
        if "acceptance" in post:  # SMC: the mean Metropolis-Hastings acceptance over the queries that moved
            acc = [float(post["acceptance"][j]) for j in range(len(queries)) if int(seat_nets[j, int(queries[j, 1])]) == net
                   and np.isfinite(post["acceptance"][j])]
            report[str(net)]["acceptance_mean"] = float(np.mean(acc)) if acc else None
    return report


def hand_reading(params_list, table, calls, offsets, seat_nets_by_auction, *, board=None, dealer=None, vul=None, at: str = "end",
                 **kwargs) -> Dict[str, Dict]:
    """The hand-reading report of auctions with known deals: every auction read by each seat (reading_queries), the posterior
    of hand_posterior (kwargs: samples, seed, temperature, precision, row_budget, method, moves, ess_threshold), scored by
    reading_stats per observer net."""
    queries, seat_nets = reading_queries(offsets, seat_nets_by_auction, dealer, at)
    post = hand_posterior(params_list, table, calls, offsets, queries, seat_nets, board=board, dealer=dealer, vul=vul, **kwargs)
    owners, _ = unpack_deal_table(table)
    return reading_stats(post, queries, seat_nets, owners, board)


def selfplay_auctions(params_a, params_b, table, n_boards: int, seed: int = 0, device="cuda"):
    """Both tables of a duplicate match of net 0 (params_a, team 1) against net 1 (params_b) on n_boards boards of `table`,
    played by the host match loop with `record=` (evaluation.make_simple_duplicate_evaluate, rng PRNGKey(seed)).  Players are
    mapped to seats from the initial state's shuffled_players; table B hands every seat to the other team.
    -> dict(calls u8, offsets i64[2n + 1], board i32, dealer i8, vul u8 (bit 0 NS, bit 1 EW), seat_nets i32[2n, 4]): auction
    2i is board i at table A, 2i + 1 at table B."""
    from . import BridgeBidding, board_log
    from . import random as brandom
    from .evaluation import make_simple_duplicate_evaluate
    env = BridgeBidding(table=np.ascontiguousarray(table, dtype=np.uint8), device=device)
    rng = brandom.PRNGKey(seed)
    _, sub = brandom.split(rng)
    state0 = env.init(env.make_keys(sub, n_boards))  # the draws the evaluator makes
    deal = state0._deal.cpu().numpy()
    dealer = state0._dealer.cpu().numpy()
    players = state0._shuffled_players.cpu().numpy()
    vul = state0._vul_NS.cpu().numpy().astype(np.uint8) | (state0._vul_EW.cpu().numpy().astype(np.uint8) << 1)
    evaluate = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n_boards)
    record = []
    evaluate(params_a, params_b, rng, record=record)
    hist_a, hist_b = board_log.split_tables(record)
    calls, offsets, nets = [], [0], []
    for i in range(n_boards):
        team_a = [int(players[i][s]) // 2 for s in range(4)]  # 0: team 1 (net 0), 1: team 2 (net 1)
        for hist, seat_net in ((hist_a[i], team_a), (hist_b[i], [1 - x for x in team_a])):
            calls.extend(hist)
            offsets.append(len(calls))
            nets.append(seat_net)
    rep = lambda a: np.repeat(np.asarray(a), 2)  # noqa: E731
    return dict(calls=np.array(calls, np.uint8), offsets=np.array(offsets, np.int64), board=rep(deal).astype(np.int32),
                dealer=rep(dealer).astype(np.int8), vul=rep(vul).astype(np.uint8), seat_nets=np.array(nets, np.int32))
