"""GPU: the bidding-system statistics (DESIGN.md f15).  Every histogram is compared by exact integer equality with
tests/system_ref.py: brl_system_stats_auctions on the golden auctions, brl_duplicate_match's histogram [21] against the host
loop's recorded auctions (with every other output bit-equal to the call without it), brl_system_stats on its own, and
evaluation.make_bidding_system_evaluate against the per-match device histograms."""
import numpy as np
import pytest
import torch

from tests import helpers as H
from tests import system_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FORCE_FUSED, FORCE_LAYERS = 1 << 30, 1 << 29  # BRL_F_TUNE_MLP_FUSED, BRL_F_TUNE_MLP_LAYERS (include/brl_b200.h)


def _counts(hist):
    from brl_b200 import ops
    return ops.system_hist_counts(hist).cpu().numpy()


def _env(rows=5000, seed=4):
    from brl_b200 import BridgeBidding
    from brl_b200.deals import synthetic_deal_table
    return BridgeBidding(table=synthetic_deal_table(rows, seed=seed), device=DEV)


# ---- brl_system_stats_auctions ------------------------------------------------------------------------------------------
def test_stored_auctions_equal_the_reference(tmp_path):
    from brl_b200 import ops, sl
    from brl_b200.deals import unpack_deal_table
    from oracle import sl_ref
    boards, gold = H.load_boards(), H.load_auctions()
    owners = unpack_deal_table(boards["table"])[0]
    want = R.auctions_hist(owners, gold["calls"].astype(np.int64), gold["offsets"], gold["board"], gold["dealer"])
    t = lambda x, dt: torch.as_tensor(np.asarray(x).astype(dt), device=DEV)  # noqa: E731
    args = (t(boards["table"], np.uint8), t(gold["calls"], np.uint8), t(gold["offsets"], np.int64))
    extra = dict(board=t(gold["board"], np.int32), dealer=t(gold["dealer"], np.int8))
    hist = ops.new_system_hist(1, DEV)
    hist.view(torch.int32).fill_(0)
    ops.system_stats_auctions(*args, hist, **extra)
    assert (_counts(hist) == want).all() and want[..., 95].sum() == len(gold["calls"])
    ops.system_stats_auctions(*args, hist, **extra)                      # += : twice the counts
    assert (_counts(hist) == 2 * want).all()
    ops.system_stats_auctions(args[0], args[1][:0], args[2][:1], hist)     # no auctions: a no-op
    assert (_counts(hist) == 2 * want).all()
    # the SL data file's trajectories: deal row t, dealer North (NULL board and dealer), through the report's reader
    g = np.load(H.os.path.join(H.GOLDEN, "sl_golden.npz"))
    traj = sl.parse_trajectories(sl_ref.write_lines(tmp_path / "golden.txt", sl_ref.golden_lines({k: g[k] for k in g.files})))
    want = R.auctions_hist(unpack_deal_table(traj.table)[0], traj.calls.astype(np.int64), traj.offsets)
    from brl_b200 import system
    assert (system.from_auctions(traj, DEV).hist == want[0]).all()
    z = dict(table=boards["table"], calls=gold["calls"], offsets=gold["offsets"], board=gold["board"], dealer=gold["dealer"])
    assert (system.from_auctions(z, DEV).hist == R.auctions_hist(owners, gold["calls"].astype(np.int64), gold["offsets"],
                                                                 gold["board"], gold["dealer"])[0]).all()


# ---- brl_duplicate_match [21] against the host loop -------------------------------------------------------------------
def _device_match(env, n, nets, models, tune=0, single_bf16=False, with_hist=True):
    from brl_b200 import ops, random as brandom
    from brl_b200.evaluation import _MatchBuffers
    from brl_b200.models import make_forward_pass
    width = len(models)
    b = _MatchBuffers(n, len(nets), 0, DEV, with_models=True, with_tables=True, players=width == 4)
    fp = make_forward_pass("relu", "DeepMind", precision="tc-bf16" if single_bf16 else None)
    size = ops._lib.load().brl_mlp_packed_bytes()
    for m, p in enumerate(nets):
        fp.pack_into(p, b.pool[m, :size])
    _, sub = brandom.split(brandom.PRNGKey(n))
    b.keys.copy_(env.make_keys(sub, n))
    b.env_models.copy_(torch.tensor(models, dtype=torch.int32, device=DEV).expand(n, width))
    hist = None
    if with_hist:
        hist = ops.new_system_hist(len(nets), DEV)
        hist.view(torch.int32).fill_(0)
    b.play(env, single_bf16, tune, hist)
    torch.cuda.synchronize()
    assert int(b.status[0]) == 0
    return b, hist


def _reference_hist(env, n, nets, models, precision, tune, monkeypatch):
    """the host loop's auctions (make_simple_duplicate_evaluate with `record`), per table, attributed by player id"""
    from brl_b200 import board_log, ops, random as brandom
    from brl_b200 import evaluation as ev
    from brl_b200.deals import unpack_deal_table
    orig = ev.make_forward_pass
    monkeypatch.setattr(ev, "make_forward_pass", lambda **kw: orig(precision=precision, **kw))
    if tune:
        orig_rows = ops.policy_act_rows
        monkeypatch.setattr(ops, "policy_act_rows", lambda *a, **kw: orig_rows(*a, **{**kw, "tune": kw.get("tune", 0) | tune}))
    host = ev.make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)
    net = lambda k: nets[k]  # noqa: E731
    if len(models) == 2:
        kw = {}
        a, b = models
    else:
        a, p1, b, p3 = models
        kw = dict(team1_partner=net(p1), team2_partner=net(p3))
    record = []
    host(net(a), net(b), brandom.PRNGKey(n), record=record, **kw)
    _, sub = brandom.split(brandom.PRNGKey(n))
    st = env.init(env.make_keys(sub, n))
    deal, dealer, players = (x.cpu().numpy() for x in (st._deal, st._dealer, st._shuffled_players))
    hist_a, hist_b = board_log.split_tables(record)
    owners = unpack_deal_table(env.table_np)[0]
    by_player = list(models) if len(models) == 4 else [models[0], models[0], models[1], models[1]]
    want = R.new_hist(len(nets))
    for i in range(n):
        pa = players[i]
        pb = pa[[1, 0, 3, 2]]                                     # table B: the seats handed to the other team
        for calls, seating in ((hist_a[i], pa), (hist_b[i], pb)):
            R.add_auction(want, owners[int(deal[i])], int(dealer[i]), calls,
                          net_of_seat=[by_player[int(seating[s])] for s in range(4)])
    return want, sum(len(h) for h in hist_a) + sum(len(h) for h in hist_b)


CASES = [("tc", 0, (0, 1)), ("tc-bf16", 0, (0, 1)), ("tc", FORCE_LAYERS, (0, 1)), ("tc", FORCE_FUSED, (0, 1)),
         ("tc", 0, (2, 0)), ("tc", 0, (0, 1, 2, 3)), ("tc-bf16", FORCE_FUSED, (3, 1, 0, 2))]


@pytest.mark.parametrize("precision, tune, models", CASES)
@pytest.mark.parametrize("n", [1, 100, 4096, 10000])
def test_match_histogram_equals_the_host_loop(n, precision, tune, models, monkeypatch):
    if n == 10000 and (precision, tune, models) not in (CASES[0], CASES[5]):
        pytest.skip("the 10,000-board host replay runs for the per-team and per-player default cases")
    env = _env()
    M = 3 if len(models) == 2 and max(models) == 2 else (2 if len(models) == 2 else 4)
    nets = [H.seeded_params(900 + k, DEV) for k in range(M)]
    single = precision == "tc-bf16"
    b, hist = _device_match(env, n, nets, models, tune, single)
    plain, _ = _device_match(env, n, nets, models, tune, single, with_hist=False)
    assert torch.equal(b.cum_return, plain.cum_return) and torch.equal(b.sums, plain.sums)
    assert torch.equal(b.status, plain.status)
    for ta, tb in zip(b.tables, plain.tables):
        for f in ("terminated", "rewards", "last_bid", "last_bidder", "call_x", "call_xx"):
            assert torch.equal(getattr(ta, f), getattr(tb, f)), f
    want, decisions = _reference_hist(env, n, nets, models, precision, tune, monkeypatch)
    got = _counts(hist)
    assert got[..., 95].sum() == decisions
    assert (got == want).all()


# ---- brl_system_stats on its own ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("by_player", [False, True])
def test_system_stats_adds_to_a_poisoned_histogram_with_done_masking(by_player):
    """random-legal auctions (brl_rollout_random's actions) stepped one call at a time; every step's decisions are counted
    from the state before it, with a random `done` mask and random nets, into a histogram pre-filled with a pattern"""
    from brl_b200 import ops
    from brl_b200.deals import unpack_deal_table
    env = _env(rows=3000, seed=9)
    n, steps, M = 3000, 24, 3
    rng = np.random.default_rng(5)
    packed = env.init(env.make_keys(3, n))._packed.clone()
    poison = torch.as_tensor(rng.integers(0, 1 << 20, (M,) + ops.SYSTEM_SHAPE), dtype=torch.int64)
    hist = poison.to(torch.int32).to(DEV).view(torch.uint32)
    env_models = torch.as_tensor(rng.integers(0, M, (n, 4 if by_player else 2)), dtype=torch.int32, device=DEV)
    owners = unpack_deal_table(env.table_np)[0]
    f0 = ops.state_fields(packed)
    deal, dealer, players = (f0[k].cpu().numpy() for k in ("deal", "dealer", "shuffled_players"))
    calls = [[] for _ in range(n)]
    masked = [set() for _ in range(n)]
    out = ops.EnvOutputs(n, DEV)
    live = np.ones(n, bool)
    mask = torch.empty((n, 38), dtype=torch.uint8, device=DEV)
    for _ in range(steps):
        ops.legal_mask(packed, mask)
        legal = mask.cpu().numpy().astype(bool)
        act = np.array([rng.choice(np.flatnonzero(legal[i])) for i in range(n)], dtype=np.int32)
        done = (rng.random(n) < 0.2) | ~live
        action = torch.as_tensor(act, device=DEV)
        ops.system_stats(packed, env.table, action, hist, done=torch.as_tensor(done.astype(np.uint8), device=DEV),
                         env_models=env_models)
        for i in np.flatnonzero(live):
            if done[i]:
                masked[i].add(len(calls[i]))
            calls[i].append(int(act[i]))
        ops.step(packed, action, env.table, packed, out)
        live &= out.terminated.cpu().numpy() == 0
    torch.cuda.synchronize()
    em = env_models.cpu().numpy()
    want = R.new_hist(M)
    for i in range(n):
        for t in range(len(calls[i])):
            if t in masked[i]:
                continue
            p = int(players[i][(int(dealer[i]) + t) % 4])
            m = int(em[i, p]) if by_player else int(em[i, 0 if p < 2 else 1])
            R.add_call(want, owners[int(deal[i])], int(dealer[i]), calls[i], t, m)
    assert (_counts(hist) - poison.numpy() == want).all()
    ops.system_stats(packed, env.table, torch.zeros(0, dtype=torch.int32, device=DEV), hist)   # an empty batch: a no-op


# ---- make_bidding_system_evaluate -------------------------------------------------------------------------------------
@pytest.mark.parametrize("opponent", [None, 1])
@pytest.mark.parametrize("max_envs", [1 << 20, 150])
def test_system_evaluate_equals_the_per_match_histograms(opponent, max_envs, tmp_path):
    import torch.distributed as dist
    from brl_b200.evaluation import make_bidding_system_evaluate
    from brl_b200 import random as brandom
    env = _env()
    n, M = 100, 3
    nets = [H.seeded_params(950 + k, DEV) for k in range(M)]
    system = make_bidding_system_evaluate(env, "relu", "DeepMind", n, max_envs=max_envs)
    got = system(nets, brandom.PRNGKey(n), opponent=opponent)
    want = R.new_hist(M)
    decisions = np.zeros(M, np.int64)
    for m in range(M):
        _, hist = _device_match(env, n, nets, (m, m if opponent is None else opponent))
        h = _counts(hist)
        want += h
        decisions += h[..., 95].reshape(M, -1).sum(axis=1)
    assert got.dtype == np.int64 and (got == want).all()
    assert (got[..., 95].reshape(M, -1).sum(axis=1) == decisions).all()
    dist.init_process_group("gloo", init_method=f"file://{tmp_path}/pg", rank=0, world_size=1)
    try:
        assert (system(nets, brandom.PRNGKey(n), opponent=opponent) == got).all()
    finally:
        dist.destroy_process_group()
