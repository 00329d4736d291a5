"""CPU: the host side of the device-resident model zoo and its PFSP probe -- the zoo's logical index <-> pool slot
bookkeeping against the host list ppo.train trims, opponent copies, packed-opponent handles, the memory budget, and the
probe's pair / range / shard layout."""
import numpy as np
import pytest
import torch


class _MarkedZoo:
    """a ModelZoo on the CPU whose packing writes the appended model's id (the real pack is a device kernel)"""

    def __new__(cls, capacity):
        from brl_b200.zoo import ModelZoo
        z = ModelZoo(capacity, "cpu")
        z._pack_into = lambda params, blob: blob[:8].copy_(torch.tensor([params], dtype=torch.int64).view(torch.uint8))
        return z


def _marker(zoo, slot):
    return int(zoo.blob(slot)[:8].view(torch.int64)[0])


@pytest.mark.parametrize("capacity", [1, 2, 3, 5])
def test_logical_index_names_the_model_of_the_trimmed_host_list(capacity):
    zoo = _MarkedZoo(capacity)
    host = []
    assert zoo.pool.shape[0] == 1 + capacity and len(zoo) == 0
    base = zoo.pool.data_ptr()
    for model in range(100, 113):
        zoo.append(model)
        host.append(model)
        host[:] = host[-capacity:]
        assert len(zoo) == len(host)
        slots = [zoo.slot(k) for k in range(len(zoo))]
        assert sorted(slots) == list(range(1, len(zoo) + 1))              # distinct slots, never the learner's slot 0
        assert [_marker(zoo, s) for s in slots] == host
        assert zoo.pool.data_ptr() == base                                 # allocated once
    zoo.set_learner(7)
    assert _marker(zoo, 0) == 7 and [_marker(zoo, zoo.slot(k)) for k in range(len(zoo))] == host


def test_an_empty_zoo_ignores_appends():
    zoo = _MarkedZoo(0)
    zoo.append(1)
    assert len(zoo) == 0 and zoo.pool.shape[0] == 1


def test_an_opponent_is_a_copy_that_outlives_its_slot():
    from brl_b200.models import PackedParams
    zoo = _MarkedZoo(2)
    zoo.append(1)
    zoo.append(2)
    opp = zoo.opponent(0)
    assert isinstance(opp, PackedParams) and opp.blob.data_ptr() != zoo.blob(zoo.slot(0)).data_ptr()
    slot = zoo.slot(0)
    zoo.append(3)                                                          # the ring reuses model 1's slot
    assert _marker(zoo, slot) == 3
    assert int(opp.blob[:8].view(torch.int64)[0]) == 1


def test_packed_params_stand_in_for_fp32_params():
    from brl_b200 import ops
    from brl_b200.models import PackedParams, make_forward_pass
    size = ops._lib.load().brl_mlp_packed_bytes()
    blob = torch.randint(0, 256, (size,), dtype=torch.uint8)
    p = PackedParams(blob)
    fp = make_forward_pass()
    assert fp._packed(p) is blob
    out = torch.zeros(ops.mlp_pool_stride(), dtype=torch.uint8)
    fp.pack_into(p, out[:size])
    assert torch.equal(out[:size], blob) and not out[size:].any()
    for bad in (blob[:-1], blob.view(torch.int8), blob.view(1, -1)):
        with pytest.raises(ValueError):
            PackedParams(bad)


def test_memory_budget(monkeypatch):
    from brl_b200 import ops, zoo
    from brl_b200.evaluation import pair_match_bytes
    stride = ops.mlp_pool_stride()
    assert zoo.device_zoo_bytes(0, 100) == stride and zoo.device_zoo_bytes(7, 0) == 8 * stride
    for K in (1, 10, 100):
        assert zoo.device_zoo_bytes(K, 100) == (1 + K) * stride + pair_match_bytes(100 * K, 1 + K, K)
    # one chunk of the probe holds at most max_envs envs, over all 1 + capacity nets
    assert zoo.device_zoo_bytes(20000, 100) == 20001 * stride + pair_match_bytes(10485 * 100, 20001, 10485)
    need = zoo.device_zoo_bytes(100, 100)
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (need + (16 << 30), 180 << 30))
    assert zoo.device_zoo_fits(100, 100, "cuda:0")
    assert not zoo.device_zoo_fits(101, 100, "cuda:0")
    assert not zoo.device_zoo_fits(100, 100, "cuda:0", reserve_bytes=(16 << 30) + 1)


class _FakeEnv:
    """what the probe reads of an env when its match op is replaced (CPU)"""
    device, table, illegal_penalty, illegal_bonus = torch.device("cpu"), None, -1.0, 1.0

    def make_keys(self, key, n, offset=0):
        return torch.arange(n, dtype=torch.int64)


def _held_bytes(bufs, pool):
    """device bytes of a buffer set, its caller-owned pool not counted"""
    ts = [bufs.keys, bufs.env_models, bufs.offsets, bufs.scratch, bufs.cum_return, bufs.sums, bufs.status]
    assert all(t.data_ptr() != pool.data_ptr() for t in ts)
    return sum(t.numel() * t.element_size() for t in ts)


@pytest.mark.parametrize("capacity,n,max_envs", [(6, 100, 1 << 20), (6, 100, 250), (5, 257, 300)])
def test_probe_holds_what_the_budget_counts_while_the_zoo_fills(capacity, n, max_envs, monkeypatch):
    """the probe's buffers are allocated once, for the whole capacity, and are exactly what device_zoo_bytes counts beside
    the pool -- before the first probe (reserve) and after every probe of a growing zoo"""
    from brl_b200 import evaluation as ev, zoo as zoo_mod
    from brl_b200 import ops
    calls = []

    def fake_play(self, eval_env, single_bf16, tune):
        assert self.scratch.numel() >= ops.duplicate_match_scratch_bytes(self.keys.shape[0], self.pool.shape[0])  # prefix fits
        calls.append((self.keys.shape[0], self.sums.shape[0]))
        self.sums.zero_()
        self.sums[:, 0] = 1.0
    monkeypatch.setattr(ev._MatchBuffers, "play", fake_play)
    zoo = _MarkedZoo(capacity)
    probe = ev.make_device_pfsp_probe(_FakeEnv(), "relu", "DeepMind", n, max_envs=max_envs)
    budget = zoo_mod.device_zoo_bytes(capacity, n, max_envs) - zoo.pool.numel()
    assert probe.buffers() is None
    probe.reserve(zoo)
    first = probe.buffers()
    ptrs = (first.keys.data_ptr(), first.scratch.data_ptr())
    assert _held_bytes(first, zoo.pool) == budget
    for K in range(1, capacity + 1):
        zoo.append(K)
        calls.clear()
        stats = probe(0, zoo, 1)
        assert len(stats) == K
        held = probe.buffers()
        assert held is first and (held.keys.data_ptr(), held.scratch.data_ptr()) == ptrs    # nothing allocated
        assert _held_bytes(held, zoo.pool) == budget
        per_chunk = max(1, max_envs // n)
        assert calls == [(min(per_chunk, K - c0) * n, min(per_chunk, K - c0)) for c0 in range(0, K, per_chunk)]


@pytest.mark.parametrize("num_pairs,n,per_chunk", [(1, 1, 1), (17, 100, 17), (17, 100, 3), (5, 257, 2), (400, 100, 10485)])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_pair_chunk_layout_shards_every_match_by_global_env_index(num_pairs, n, per_chunk, world):
    from brl_b200.dist import shard_range
    from brl_b200.evaluation import pair_chunk_layout
    seen = np.zeros((num_pairs, n), dtype=np.int64)
    chunks = None
    for rank in range(world):
        layout = list(pair_chunk_layout(num_pairs, n, per_chunk, rank, world))
        starts = [c[0] for c in layout]
        assert chunks is None or starts == chunks                          # every rank walks the same chunks
        chunks = starts
        assert starts == list(range(0, num_pairs, per_chunk))
        for c0, P, lo, hi, p_lo, p_hi, bounds in layout:
            assert P == min(per_chunk, num_pairs - c0) and (lo, hi) == shard_range(P * n, rank, world)
            if hi == lo:
                continue
            assert bounds[0] == 0 and bounds[-1] == hi - lo and (np.diff(bounds) >= 0).all()
            for p in range(p_lo, p_hi):                                    # local range of match p: its boards, in order
                g = lo + np.arange(bounds[p - p_lo], bounds[p - p_lo + 1])
                assert (g // n == p).all()
                seen[c0 + p, g % n] += 1
    assert (seen == 1).all()
