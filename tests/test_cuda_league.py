"""GPU: the self-play league (workspace/eval_selfplay_league.py) -- brl_model_rows, the grouped forward over a pool of nets
(brl_policy_act_grouped) against the one-net listed forward, the batched tournament against pairwise
make_simple_duplicate_evaluate matches (both precisions, one chunk and several), the golden seeded match, and the XLA symbols of
the new ops."""
import ctypes as C
import itertools

import numpy as np
import pytest
import torch

from tests import helpers as H
from tests.test_cuda_xla import _call_xla

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FORCE_FUSED, FORCE_LAYERS = 1 << 30, 1 << 29  # BRL_F_TUNE_MLP_FUSED, BRL_F_TUNE_MLP_LAYERS (include/brl_b200.h)


def _obs_and_mask(n, seed=11, steps=9):
    from brl_b200 import ops
    from brl_b200.deals import synthetic_deal_table
    table = torch.as_tensor(synthetic_deal_table(500, 2), device=DEV)
    state, out = ops.new_state(n, DEV), ops.EnvOutputs(n, DEV, torch.bfloat16)
    ops.init(ops.make_keys(seed, n, DEV), table, state, out)
    for i in range(steps):
        ops.step(state, None, table, state, out, autoreset=True, random_action=True, seed=seed, step_index=i)
    return out.observation, out.legal_action_mask


def _grouping(sizes, n_done, seed):
    """players, done and env_models with exactly sizes[m] live envs acting with net m (shuffled), n_done finished envs"""
    M = len(sizes)
    g = np.random.default_rng(seed)
    acting = np.concatenate([np.full(s, m) for m, s in enumerate(sizes)] + [g.integers(0, M, n_done)]).astype(np.int32)
    done = np.concatenate([np.zeros(sum(sizes)), np.ones(n_done)]).astype(np.uint8)
    perm = g.permutation(acting.shape[0])
    acting, done = acting[perm], done[perm]
    player = g.integers(0, 4, acting.shape[0]).astype(np.int8)
    env_models = g.integers(0, M, (acting.shape[0], 2)).astype(np.int32)
    env_models[np.arange(acting.shape[0]), (player >= 2).astype(int)] = acting
    t = lambda a: torch.as_tensor(a, device=DEV).contiguous()  # noqa: E731
    return t(player), t(done), t(env_models), acting, done


CASES = [  # (M, group sizes): totals below and above 4096 padded rows, groups of 0, 1, 127, 128, 129 and thousands
    (1, [129]),
    (3, [0, 1, 127]),
    (3, [128, 129, 5000]),
    (17, [0, 1, 127, 128, 129, 0, 3, 0, 0, 0, 2, 0, 0, 0, 0, 0, 1]),
    (17, [0, 1, 127, 128, 129, 3000, 7, 255, 256, 257, 0, 64, 2, 999, 0, 1, 4500]),
]


@pytest.mark.parametrize("single_bf16", [False, True])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_grouped_forward_equals_per_model_listed_forward(case, single_bf16):
    from brl_b200 import ops
    from brl_b200.models import make_forward_pass
    M, sizes = CASES[case]
    player, done, env_models, acting, done_np = _grouping(sizes, n_done=300, seed=case)
    n = player.shape[0]
    obs, mask = _obs_and_mask(n, seed=case + 3)
    fp = make_forward_pass(precision="tc-bf16" if single_bf16 else "tc")
    nets = [H.seeded_params(100 + m, DEV) for m in range(M)]
    pool = ops.mlp_pack_pool(nets, fp.pack_into)
    cap = ops.model_rows_capacity(n, M)
    rows = torch.full((cap,), -7, dtype=torch.int32, device=DEV)
    block_model = torch.full((cap // 256,), -7, dtype=torch.int32, device=DEV)
    counts = torch.empty(M, dtype=torch.int32, device=DEV)
    offsets = torch.empty(M + 1, dtype=torch.int32, device=DEV)
    ops.model_rows(player, done, env_models, rows, counts, offsets, block_model)
    # the grouping: counts, padded offsets, each group's envs then -1 padding, the block -> net map
    assert counts.tolist() == sizes
    padded = [(s + 255) // 256 * 256 for s in sizes]
    off = offsets.tolist()
    assert off == [0] + list(np.cumsum(padded))
    for m in range(M):
        grp = rows[off[m]:off[m + 1]].cpu().numpy()
        assert sorted(grp[:sizes[m]].tolist()) == np.nonzero((acting == m) & (done_np == 0))[0].tolist()
        assert (grp[sizes[m]:] == -1).all()
        assert (block_model[off[m] // 256:off[m + 1] // 256].cpu().numpy() == m).all()
    n_rows = off[M]
    tune = FORCE_FUSED if n_rows >= 4096 else FORCE_LAYERS  # the path the grouped call takes, forced on the one-net calls
    action = torch.full((n,), -5, dtype=torch.int32, device=DEV)
    logits = torch.full((n, 38), 7.0, dtype=torch.float32, device=DEV)
    scratch = torch.empty(ops.policy_grouped_scratch_bytes(n, M), dtype=torch.uint8, device=DEV)
    ops.policy_act_grouped(obs, pool, scratch, mask, action, rows[:n_rows], block_model, logits, n_rows=offsets[M:],
                           single_bf16=single_bf16)
    a_ref = torch.full((n,), -5, dtype=torch.int32, device=DEV)
    lg_ref = torch.full((n, 38), 7.0, dtype=torch.float32, device=DEV)
    for m in range(M):
        listed = rows[off[m]:off[m] + sizes[m]].contiguous()
        if sizes[m]:
            ops.policy_act_rows(obs, fp._packed(nets[m]), ops.mlp_rows_scratch(sizes[m], DEV), mask, a_ref, listed, logits=lg_ref,
                                single_bf16=single_bf16, tune=tune)
    assert torch.equal(action, a_ref) and torch.equal(logits, lg_ref)
    unlisted = torch.as_tensor(done_np, device=DEV) != 0
    assert bool((action[unlisted] == -5).all()) and bool((logits[unlisted] == 7.0).all())
    assert bool(mask[~unlisted].gather(1, action[~unlisted].long()[:, None]).all())
    # the mask and logits are optional, and without n_rows the rows end at the count
    a2 = torch.full((n,), -5, dtype=torch.int32, device=DEV)
    ops.policy_act_grouped(obs, pool, scratch, mask, a2, rows[:n_rows], block_model, single_bf16=single_bf16)
    assert torch.equal(a2, a_ref)


def test_grouped_forward_rejects_sampling():
    from brl_b200 import _lib, ops
    rows = torch.zeros(256, dtype=torch.int32, device=DEV)
    obs = torch.zeros((4, 480), dtype=torch.bfloat16, device=DEV)
    pool = torch.zeros((1, ops.mlp_pool_stride()), dtype=torch.uint8, device=DEV)
    scratch = torch.empty(ops.policy_grouped_scratch_bytes(4, 1), dtype=torch.uint8, device=DEV)
    with pytest.raises(_lib.BrlError, match="sampling"):
        ops.policy_act_grouped(obs, pool, scratch, None, torch.zeros(4, dtype=torch.int32, device=DEV), rows,
                               torch.zeros(1, dtype=torch.int32, device=DEV), tune=_lib.F_SAMPLE)


def test_grouped_forward_validates_the_row_count_tensor():
    from brl_b200 import _lib, ops
    rows, block_model = torch.zeros(256, dtype=torch.int32, device=DEV), torch.zeros(1, dtype=torch.int32, device=DEV)
    obs = torch.zeros((4, 480), dtype=torch.bfloat16, device=DEV)
    pool = torch.zeros((1, ops.mlp_pool_stride()), dtype=torch.uint8, device=DEV)
    scratch = torch.empty(ops.policy_grouped_scratch_bytes(4, 1), dtype=torch.uint8, device=DEV)
    for bad in (torch.full((1,), 256, dtype=torch.int64, device=DEV), torch.empty(0, dtype=torch.int32, device=DEV),
                torch.full((1,), 256, dtype=torch.int32)):
        with pytest.raises(_lib.BrlError, match="n_rows"):
            ops.policy_act_grouped(obs, pool, scratch, None, torch.zeros(4, dtype=torch.int32, device=DEV), rows, block_model,
                                   n_rows=bad)


@pytest.mark.parametrize("single_bf16", [False, True])
@pytest.mark.parametrize("tune", [FORCE_FUSED, FORCE_LAYERS], ids=["fused", "layers"])
@pytest.mark.parametrize("case", [2, 3])
def test_grouped_forward_sized_past_the_row_count_equals_the_call_sized_for_it(case, tune, single_bf16):
    """The device match loops size the grouped forward for the grouping's capacity and leave the padded row count in device
    memory.  A rows buffer longer than offsets[M], padded with -1, gives the actions and logits of the call whose rows end at
    the count; so does one that lists finished envs past the count, which must not be forwarded."""
    from brl_b200 import ops
    from brl_b200.models import make_forward_pass
    M, sizes = CASES[case]
    player, done, env_models, _, done_np = _grouping(sizes, n_done=300, seed=case)
    n = player.shape[0]
    obs, mask = _obs_and_mask(n, seed=case + 3)
    fp = make_forward_pass(precision="tc-bf16" if single_bf16 else "tc")
    pool = ops.mlp_pack_pool([H.seeded_params(100 + m, DEV) for m in range(M)], fp.pack_into)
    cap = ops.model_rows_capacity(n, M)
    rows = torch.full((cap,), -7, dtype=torch.int32, device=DEV)
    block_model = torch.full((cap // 256,), -7, dtype=torch.int32, device=DEV)
    counts, offsets = torch.empty(M, dtype=torch.int32, device=DEV), torch.empty(M + 1, dtype=torch.int32, device=DEV)
    ops.model_rows(player, done, env_models, rows, counts, offsets, block_model)
    n_rows, long = int(offsets[M]), int(offsets[M]) + 16 * 256

    def run(rows_buf, blocks_buf):
        action = torch.full((n,), -5, dtype=torch.int32, device=DEV)
        logits = torch.full((n, 38), 7.0, dtype=torch.float32, device=DEV)
        ops.policy_act_grouped(obs, pool, ops.mlp_rows_scratch(rows_buf.shape[0], DEV), mask, action, rows_buf, blocks_buf,
                               logits, n_rows=offsets[M:], single_bf16=single_bf16, tune=tune)
        return action, logits

    a_ref, lg_ref = run(rows[:n_rows], block_model[:n_rows // 256])
    assert bool((a_ref >= 0).sum() == sum(sizes))
    rows_long = torch.full((long,), -1, dtype=torch.int32, device=DEV)
    rows_long[:n_rows] = rows[:n_rows]
    blocks_long = torch.zeros(long // 256, dtype=torch.int32, device=DEV)   # valid net ids past the count
    blocks_long[:n_rows // 256] = block_model[:n_rows // 256]
    a, lg = run(rows_long, blocks_long)
    assert torch.equal(a, a_ref) and torch.equal(lg, lg_ref)
    finished = torch.nonzero(torch.as_tensor(done_np, device=DEV)).flatten().to(torch.int32)
    rows_long[n_rows:] = finished.repeat(-(-(long - n_rows) // finished.shape[0]))[:long - n_rows]
    a, lg = run(rows_long, blocks_long)
    assert torch.equal(a, a_ref) and torch.equal(lg, lg_ref)


def _script_matrices(M, imps):
    """workspace/eval_selfplay_league.py's loop body, restated"""
    win_lose, win_lose_dis, win_lose_clip = np.zeros((M, M)), np.zeros((M, M)), np.zeros((M, M))
    for match in itertools.combinations(range(M), 2):
        imp = imps[match]
        win_lose[match[0]][match[1]] = -imp
        win_lose[match[1]][match[0]] = imp
        clip_imp = np.clip(imp, -1, 1)
        win_lose_clip[match[0]][match[1]] = -clip_imp
        win_lose_clip[match[1]][match[0]] = clip_imp
        if imp > 0:
            win_lose_dis[match[0]][match[1]] = -1
            win_lose_dis[match[1]][match[0]] = 1
        elif imp < 0:
            win_lose_dis[match[0]][match[1]] = 1
            win_lose_dis[match[1]][match[0]] = -1
    return win_lose, win_lose_dis, win_lose_clip


def _assert_league_equals_pairwise_matches(nets, num_eval_envs, max_envs, key):
    from brl_b200 import BridgeBidding
    from brl_b200.deals import synthetic_deal_table
    from brl_b200.evaluation import make_selfplay_league_evaluate, make_simple_duplicate_evaluate
    env = BridgeBidding(table=synthetic_deal_table(5000, seed=4), device=DEV)
    M = len(nets)
    league = make_selfplay_league_evaluate(env, "relu", "DeepMind", num_eval_envs, max_envs=max_envs)
    got = {}
    stats, wl, dis, clip = league(nets, key, cum_returns=got)
    match = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", num_eval_envs)
    assert list(stats) == list(itertools.combinations(range(M), 2))
    imps = {}
    for (i, j), s in stats.items():
        (mean, se, win), _, _, cum = match(nets[i], nets[j], key)
        assert torch.equal(got[(i, j)], cum), (i, j)
        assert s == (mean, se, win), (i, j)     # integer IMP sums: the statistics are the same numbers
        imps[(i, j)] = mean
    for a, b in zip((wl, dis, clip), _script_matrices(M, imps)):
        np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("num_eval_envs", [100, 1000])
def test_tournament_equals_pairwise_matches(num_eval_envs):
    from brl_b200 import random as brandom
    nets = [H.seeded_params(200 + m, DEV) for m in range(5)]
    _assert_league_equals_pairwise_matches(nets, num_eval_envs, 3 * num_eval_envs, brandom.PRNGKey(7))  # 4 chunks


LEAGUES = [  # (M, boards per match, max_envs, single_bf16): padded live totals above 4096 at the start and below it later
    (2, 5000, 1 << 20, False),
    (3, 1000, 3000, False),
    (3, 1000, 3000, True),
    (17, 100, 3000, False),
    (17, 100, 3000, True),
]


@pytest.mark.parametrize("case", range(len(LEAGUES)))
def test_tournament_equals_pairwise_matches_at_both_precisions(case, monkeypatch):
    """both the league and the pairwise matches run the precision of the case"""
    from brl_b200 import random as brandom
    import brl_b200.evaluation as ev
    M, n, max_envs, single_bf16 = LEAGUES[case]
    orig = ev.make_forward_pass
    monkeypatch.setattr(ev, "make_forward_pass", lambda **kw: orig(precision="tc-bf16" if single_bf16 else "tc", **kw))
    nets = [H.seeded_params(500 + m, DEV) for m in range(M)]
    _assert_league_equals_pairwise_matches(nets, n, max_envs, brandom.PRNGKey(11 + case))


def test_tournament_reproduces_the_golden_seeded_match():
    """pair (0, 1) of a three-net league over the 1,000 real boards is the configs[0] match of c1_seeded_match.npz"""
    from brl_b200 import BridgeBidding, random as brandom
    from brl_b200.evaluation import make_selfplay_league_evaluate
    g = H.load_c1_seeded()
    env = BridgeBidding(table=H.load_boards()["table"], device=DEV)
    nets = [H.seeded_params(int(s), DEV) for s in g["weight_seeds"]] + [H.seeded_params(3, DEV)]
    league = make_selfplay_league_evaluate(env, "relu", "DeepMind", int(g["n"]))
    got = {}
    stats, *_ = league(nets, brandom.PRNGKey(int(g["seed"])), cum_returns=got)
    assert (got[(0, 1)].cpu().numpy() == g["imps"]).all()
    np.testing.assert_allclose(stats[(0, 1)], g["stats"], rtol=1e-9, atol=1e-12)


def test_match_stats_ranges_equal_match_stats_on_each_slice():
    from brl_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randint(-24, 25, (50_000,), generator=g, device=DEV).to(torch.float32)
    bounds = [0, 0, 1, 100, 357, 20_000, 20_001, 50_000]
    offs = torch.tensor(bounds, dtype=torch.int64, device=DEV)
    sums = torch.zeros((len(bounds) - 1, 8), dtype=torch.float64, device=DEV)
    ops.match_stats_ranges(x, offs, sums)
    for p in range(len(bounds) - 1):
        ref = torch.zeros(8, dtype=torch.float64, device=DEV)
        if bounds[p + 1] > bounds[p]:
            ops.match_stats(x[bounds[p]:bounds[p + 1]].contiguous(), ref)
        assert torch.equal(sums[p], ref), p


def test_league_xla_symbols_equal_direct_ops_and_empty_batches_are_no_ops():
    from brl_b200 import _lib, ops
    from brl_b200.models import make_forward_pass
    M, sizes = CASES[2]
    player, done, env_models, _, _ = _grouping(sizes, n_done=50, seed=9)
    n = player.shape[0]
    cap = ops.model_rows_capacity(n, M)
    out = [[torch.full((k,), -3, dtype=torch.int32, device=DEV) for k in (cap, M, M + 1, cap // 256)] for _ in range(2)]
    ops.model_rows(player, done, env_models, *out[0])
    _call_xla("brl_model_rows", [player, done, env_models, *out[1]], ops._params(n, k_steps=M))
    torch.cuda.synchronize()
    for a, b in zip(*out):
        assert torch.equal(a.sort().values, b.sort().values)   # rows inside a group come in arrival order
    assert torch.equal(out[0][2], out[1][2]) and torch.equal(out[0][3], out[1][3])
    rows, block_model, n_rows = out[0][0], out[0][3], int(out[0][2][M])
    obs, mask = _obs_and_mask(n)
    pool = ops.mlp_pack_pool([H.seeded_params(300 + m, DEV) for m in range(M)], make_forward_pass().pack_into)
    scratch = torch.empty(ops.policy_grouped_scratch_bytes(n, M), dtype=torch.uint8, device=DEV)
    acts = [torch.full((n,), -5, dtype=torch.int32, device=DEV) for _ in range(2)]
    lgs = [torch.full((n, 38), 7.0, dtype=torch.float32, device=DEV) for _ in range(2)]
    ops.policy_act_grouped(obs, pool, scratch, mask, acts[0], rows[:n_rows], block_model, lgs[0], n_rows=out[0][2][M:])
    _call_xla("brl_policy_act_grouped", [obs, pool, scratch, mask, acts[1], rows[:n_rows].contiguous(), block_model, lgs[1],
                                         out[0][2][M:]], ops._params(n_rows, k_steps=M))
    torch.cuda.synchronize()
    assert torch.equal(acts[0], acts[1]) and torch.equal(lgs[0], lgs[1])
    x = torch.arange(1000, device=DEV, dtype=torch.float32) % 7 - 3
    offs = torch.tensor([0, 10, 999, 1000], dtype=torch.int64, device=DEV)
    sums = [torch.zeros((3, 8), dtype=torch.float64, device=DEV) for _ in range(2)]
    ops.match_stats_ranges(x, offs, sums[0])
    _call_xla("brl_match_stats_ranges", [x, offs, sums[1]], ops._params(3))
    torch.cuda.synchronize()
    assert torch.equal(sums[0], sums[1])
    # empty batches: NULL buffers, BRL_OK; brl_model_rows reports empty groups
    L = _lib.load()
    nulls = (C.c_void_p * 8)()
    stream = torch.cuda.current_stream().cuda_stream
    for name in ("brl_model_rows", "brl_policy_act_grouped", "brl_match_stats_ranges"):
        p0 = ops._params(0, k_steps=M)
        assert getattr(L, name)(C.c_void_p(stream), nulls, C.byref(p0), C.sizeof(p0)) == 0, name
    counts, offsets = torch.full((M,), 9, dtype=torch.int32, device=DEV), torch.full((M + 1,), 9, dtype=torch.int32, device=DEV)
    e = torch.empty(0, dtype=torch.int32, device=DEV)
    ops.model_rows(torch.empty(0, dtype=torch.int8, device=DEV), None, torch.empty((0, 2), dtype=torch.int32, device=DEV), e,
                   counts, offsets, e)
    assert counts.tolist() == [0] * M and offsets.tolist() == [0] * (M + 1)
    torch.cuda.synchronize()


def test_match_stats_ranges_beyond_the_grid_limit():
    """more ranges than a grid dimension holds (65,535): the kernel strides over them; a league chunk of many small
    matches passes that many"""
    from brl_b200 import ops
    P = 70_001
    g = torch.Generator(device=DEV).manual_seed(5)
    lengths = torch.randint(0, 6, (P,), generator=g, device=DEV)
    offs = torch.zeros(P + 1, dtype=torch.int64, device=DEV)
    offs[1:] = torch.cumsum(lengths, 0)
    n = int(offs[-1])
    x = torch.randint(-24, 25, (n,), generator=g, device=DEV).to(torch.float32)
    sums = torch.zeros((P, 8), dtype=torch.float64, device=DEV)
    ops.match_stats_ranges(x, offs, sums)
    seg = torch.repeat_interleave(torch.arange(P, device=DEV), lengths)
    xd = x.double()
    want = torch.zeros((P, 8), dtype=torch.float64, device=DEV)
    for k, v in enumerate((torch.ones_like(xd), xd, xd * xd, (xd > 0).double())):
        want[:, k].index_add_(0, seg, v)
    assert torch.equal(sums, want)   # integer-valued: exact in any order


def test_model_rows_reports_an_out_of_range_net_id():
    from brl_b200 import ops
    M = 3
    player, done, env_models, _, done_np = _grouping([5, 0, 300], n_done=20, seed=4)
    n = player.shape[0]
    cap = ops.model_rows_capacity(n, M)
    out = [torch.empty(k, dtype=torch.int32, device=DEV) for k in (cap, M, M + 1, cap // 256)]
    live, dead = int(np.nonzero(done_np == 0)[0][7]), int(np.nonzero(done_np != 0)[0][3])
    bad = env_models.clone()
    bad[dead] = M                       # a finished env's id is never read
    ops.model_rows(player, done, bad, *out)
    assert out[2].tolist() == [0, 256, 256, 768]
    bad[live] = M                       # the acting net of a live env is out of range
    ops.model_rows(player, done, bad, *out)
    assert int(out[2][M]) == -1
    bad[live] = -1
    ops.model_rows(player, done, bad, *out)
    assert int(out[2][M]) == -1
    ops.model_rows(player, done, env_models, *out)   # the next call starts clean
    assert out[2].tolist() == [0, 256, 256, 768]


@pytest.mark.parametrize("world", [2, 3])
def test_league_result_does_not_depend_on_the_rank_count(world, monkeypatch):
    """the chunk's envs shard by global index: the ranks' shards (which split matches mid-way here) put together give the
    one-rank per-env returns and, summed, the one-rank statistics sums bit for bit"""
    from brl_b200 import BridgeBidding, dist as bdist, random as brandom
    from brl_b200.deals import synthetic_deal_table
    from brl_b200.evaluation import make_selfplay_league_evaluate
    env = BridgeBidding(table=synthetic_deal_table(3000, seed=6), device=DEV)
    nets = [H.seeded_params(400 + m, DEV) for m in range(4)]
    key = brandom.PRNGKey(3)
    stats_from_sums = bdist.stats_from_sums

    def run(rank, w):
        recorded, got = [], {}
        monkeypatch.setattr(bdist, "rank_world", lambda: (rank, w))
        monkeypatch.setattr(bdist, "allreduce_sums", lambda s: recorded.append(s.clone()) or s)
        # without the all-reduce a rank may hold no env of a match: its (partial) statistics are not formed then
        monkeypatch.setattr(bdist, "stats_from_sums", lambda s: stats_from_sums(s) if float(s[0]) > 0 else (0.0, 0.0, 0.0))
        league = make_selfplay_league_evaluate(env, "relu", "DeepMind", 100, max_envs=150)
        league(nets, key, cum_returns=got)
        return torch.cat(recorded), got   # sums in pair order: chunks are consecutive runs of the pairs

    ref_sums, ref_ret = run(0, 1)
    shards = [run(r, world) for r in range(world)]
    assert torch.equal(sum(s for s, _ in shards), ref_sums)
    for pair, want in ref_ret.items():
        parts = [got[pair] for _, got in shards if pair in got]
        assert torch.equal(torch.cat(parts), want), pair
