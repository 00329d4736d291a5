"""GPU: counterfactual call values (DESIGN.md f16).  brl_call_values' records are compared bit for bit with the host loop of
tests/call_values_ref.py, its sums exactly with the reference reduction of the records, and the evaluator across chunkings
and under a process group."""
import numpy as np
import pytest
import torch

from tests import call_values_ref as R
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FORCE_FUSED, FORCE_LAYERS = 1 << 30, 1 << 29  # BRL_F_TUNE_MLP_FUSED, BRL_F_TUNE_MLP_LAYERS (include/brl_b200.h)


def _env(rows=5000, seed=4):
    from brl_b200 import BridgeBidding
    from brl_b200.deals import synthetic_deal_table
    return BridgeBidding(table=synthetic_deal_table(rows, seed=seed), device=DEV)


class _Run:
    """the base match (brl_duplicate_match with Table_infos) and brl_call_values on the same keys and nets"""

    def __init__(self, env, n, nets, models, tune=0, single=False, capacity=None, poison=False, key=None):
        from brl_b200 import ops, random as brandom
        from brl_b200.evaluation import _MatchBuffers
        from brl_b200.models import make_forward_pass
        M, width = len(nets), len(models)
        b = _MatchBuffers(n, M, 0, DEV, with_models=True, with_tables=True, players=width == 4)
        fp = make_forward_pass("relu", "DeepMind", precision="tc-bf16" if single else None)
        size = ops._lib.load().brl_mlp_packed_bytes()
        for m, p in enumerate(nets):
            fp.pack_into(p, b.pool[m, :size])
        _, sub = brandom.split(key if key is not None else brandom.PRNGKey(n))
        b.keys.copy_(env.make_keys(sub, n))
        b.env_models.copy_(torch.tensor(models, dtype=torch.int32, device=DEV).expand(n, width))
        b.play(env, single, tune)
        self.match = b
        fill = (lambda t: t.fill_(-1)) if poison else (lambda t: t.zero_())
        self.gain = fill(torch.empty((M,) + ops.CALL_GAIN_SHAPE, dtype=torch.int64, device=DEV))
        self.regret = fill(torch.empty((M,) + ops.CALL_REGRET_SHAPE, dtype=torch.int64, device=DEV))
        self.mismatch = fill(torch.empty(M, dtype=torch.int64, device=DEV))
        self.status = torch.full((1,), -1 if poison else 0, dtype=torch.int32, device=DEV)
        self.records = ops.CallValueRecords(capacity if capacity is not None else 48 * n, DEV)
        if poison:
            for f in ops.CALL_RECORD_FIELDS:
                getattr(self.records, f).fill_(-1)
            self.records.r.fill_(-1.0)
            self.records.count.fill_(-1)
        self.scratch = torch.full((ops.call_values_scratch_bytes(n, M),), 0xFF if poison else 0, dtype=torch.uint8, device=DEV)
        ops.call_values(b.keys, env.table, b.pool, b.env_models, b.tables[0].rewards, b.tables[1].rewards, self.scratch,
                        self.gain, self.regret, self.mismatch, self.status, records=self.records, single_bf16=single, tune=tune)
        torch.cuda.synchronize()
        assert int(b.status[0]) == 0

    def recs(self):
        from brl_b200 import ops
        k = min(int(self.records.count[0]), self.records.capacity)
        return {f: getattr(self.records, f)[:k].cpu().numpy() for f in ops.CALL_RECORD_FIELDS + ("r",)}

    def base(self):
        return self.match.tables[0].rewards[:, 0].cpu().numpy(), self.match.tables[1].rewards[:, 0].cpu().numpy()


def _by_env_table(rec):
    """per (env, table): the indices of its records"""
    out = {}
    for k in range(len(rec["env"])):
        out.setdefault((int(rec["env"][k]), int(rec["table"][k])), []).append(k)
    return out


def _compare(dev_rec, ref_rec):
    """bit-equal records: the same decisions per (env, table), each with the same player, net, context, played call and r"""
    d, r = _by_env_table(dev_rec), _by_env_table(ref_rec)
    assert d.keys() == r.keys()
    for key, rk in r.items():
        dk = d[key]
        assert len(dk) == len(rk), key
        # one env's decisions come from successive base iterations, whose gain kernels run in order: its records' slots
        # rise in play order
        for a, b in zip(sorted(dk), rk):
            for f in ("player", "net", "context", "played"):
                assert dev_rec[f][a] == ref_rec[f][b], (key, f)
            assert np.array_equal(dev_rec["r"][a].view(np.uint32), ref_rec["r"][b].view(np.uint32)), key


CASES = [("tc", FORCE_LAYERS, (0, 1)), ("tc", FORCE_FUSED, (0, 1)), ("tc-bf16", FORCE_FUSED, (0, 1)),
         ("tc-bf16", FORCE_LAYERS, (2, 0)), ("tc", FORCE_FUSED, (0, 1, 2, 3)), ("tc", 0, (0, 1))]


@pytest.mark.parametrize("precision, tune, models", CASES)
@pytest.mark.parametrize("n", [1, 7, 100, 1000])
def test_records_and_sums_equal_the_host_loop(n, precision, tune, models):
    from brl_b200 import random as brandom
    if n == 1000 and (precision, tune, models) not in (CASES[0], CASES[4]):
        pytest.skip("the 1,000-board host replay runs for one per-team and one per-player case")
    env = _env()
    M = 3 if models == (2, 0) else len(models)
    nets = [H.seeded_params(700 + k, DEV) for k in range(M)]
    run = _Run(env, n, nets, models, tune, precision == "tc-bf16")
    assert int(run.status[0]) == 0
    got = run.recs()
    assert int(run.records.count[0]) == len(got["env"])
    ref, R_a, R_b = R.host_records(env, nets, models, n, brandom.PRNGKey(n), precision, tune)
    da, db = run.base()
    assert np.array_equal(da, R_a) and np.array_equal(db, R_b)          # the base match is the host loop's match
    _compare(got, ref)
    gain, reg, mismatch = R.reduce_records(got, da, db, M)
    assert (run.gain.cpu().numpy() == gain).all() and (run.regret.cpu().numpy() == reg).all()
    assert (run.mismatch.cpu().numpy() == mismatch).all()
    if tune:
        assert int(run.mismatch.sum()) == 0                               # pinned forward: the played branch is the game
    assert (reg[..., 1] >= 0).all() and gain[..., 0].sum() == np.isfinite(got["r"]).sum()


def test_poisoned_outputs_capacity_and_empty_batch():
    from brl_b200 import ops
    env = _env()
    nets = [H.seeded_params(710 + k, DEV) for k in range(2)]
    clean = _Run(env, 100, nets, (0, 1), FORCE_FUSED)
    poisoned = _Run(env, 100, nets, (0, 1), FORCE_FUSED, poison=True)
    for f in ("gain", "regret", "mismatch", "status"):
        assert torch.equal(getattr(clean, f), getattr(poisoned, f)), f
    _compare(poisoned.recs(), clean.recs())
    small = _Run(env, 100, nets, (0, 1), FORCE_FUSED, capacity=10)
    assert int(small.status[0]) == ops._lib.MATCH_RECORD_CAPACITY
    assert int(small.records.count[0]) == int(clean.records.count[0])
    for f in ("gain", "regret", "mismatch"):
        assert torch.equal(getattr(clean, f), getattr(small, f)), f
    e = torch.zeros(0, dtype=torch.int64, device=DEV)
    ops.call_values(e, env.table, clean.match.pool, torch.zeros((0, 2), dtype=torch.int32, device=DEV),
                    torch.zeros((0, 4), device=DEV), torch.zeros((0, 4), device=DEV), clean.scratch, clean.gain, clean.regret,
                    clean.mismatch, clean.status)                           # an empty batch: a no-op
    torch.cuda.synchronize()
    assert int(clean.status[0]) == 0 and torch.equal(clean.gain, poisoned.gain)


def test_null_required_buffer_is_a_buffer_error():
    from brl_b200 import _lib, ops
    env = _env()
    nets = [H.seeded_params(720 + k, DEV) for k in range(2)]
    run = _Run(env, 10, nets, (0, 1), FORCE_FUSED)
    b = run.match
    bufs = [ops._ptr(x) for x in (b.keys, env.table, b.pool, b.env_models, b.tables[0].rewards, b.tables[1].rewards, run.scratch,
                                  run.gain, run.regret, run.mismatch, run.status)] + [None] * 8
    for k in range(11):
        bad = list(bufs)
        bad[k] = None
        with pytest.raises(_lib.BrlError, match="NULL"):
            _lib.call("brl_call_values", torch.cuda.current_stream().cuda_stream, bad,
                      ops._params(10, k_steps=2, n_deals=env.table.shape[0]))


def test_duplicate_match_is_unchanged_by_call_values():
    env = _env()
    nets = [H.seeded_params(730 + k, DEV) for k in range(2)]
    before = _Run(env, 100, nets, (0, 1), FORCE_FUSED).match
    cum, sums = before.cum_return.clone(), before.sums.clone()
    infos = [t.rewards.clone() for t in before.tables]
    before.play(env, False, FORCE_FUSED)
    torch.cuda.synchronize()
    assert torch.equal(before.cum_return, cum) and torch.equal(before.sums, sums)
    assert all(torch.equal(t.rewards, r) for t, r in zip(before.tables, infos))


@pytest.mark.parametrize("opponent", [None, 1])
def test_evaluate_is_independent_of_chunks_and_ranks(opponent, tmp_path):
    import torch.distributed as dist
    from brl_b200 import random as brandom
    from brl_b200.evaluation import make_call_values_evaluate
    env = _env()
    n, M = 60, 3
    nets = [H.seeded_params(740 + k, DEV) for k in range(M)]
    one = make_call_values_evaluate(env, "relu", "DeepMind", n, tune=FORCE_FUSED)(nets, brandom.PRNGKey(3), opponent, True)
    many = make_call_values_evaluate(env, "relu", "DeepMind", n, max_envs=38 * 25,
                                     tune=FORCE_FUSED)(nets, brandom.PRNGKey(3), opponent, True)
    for f in ("gain_sums", "regret_sums", "mismatch"):
        assert (one[f] == many[f]).all(), f
    assert int(one["mismatch"].sum()) == 0
    assert len(one["records"]["env"]) == len(many["records"]["env"]) == int(one["regret_sums"][..., 0].sum())
    # per match: the op on that match alone gives the same sums
    want = [np.zeros_like(one[f]) for f in ("gain_sums", "regret_sums", "mismatch")]
    for m in range(M):
        run = _Run(env, n, nets, (m, m if opponent is None else opponent), FORCE_FUSED, key=brandom.PRNGKey(3))
        for w, x in zip(want, (run.gain, run.regret, run.mismatch)):
            w += x.cpu().numpy()
    assert all((w == one[f]).all() for w, f in zip(want, ("gain_sums", "regret_sums", "mismatch")))
    dist.init_process_group("gloo", init_method=f"file://{tmp_path}/pg", rank=0, world_size=1)
    try:
        again = make_call_values_evaluate(env, "relu", "DeepMind", n, tune=FORCE_FUSED)(nets, brandom.PRNGKey(3), opponent)
    finally:
        dist.destroy_process_group()
    assert all((again[f] == one[f]).all() for f in ("gain_sums", "regret_sums", "mismatch"))
