"""CPU: the host side of brl_duplicate_match (a whole duplicate match as one device-resident call) -- its XLA layout, lazy
binding, argument validation, scratch-size query, and scripts/duplicate_eval.py's arguments."""
import ctypes
import os

import pytest
import torch


def _bind(L):
    fn = L.brl_duplicate_match
    fn.restype, fn.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]
    return fn


def _params(n, M, P=0, n_deals=100, flags=0):
    from brl_b200 import _lib
    return _lib.BrlParams(n, 0, 0, 0, n_deals, flags, P, M, -1.0, 1.0, 0.0, 0.0)   # step = P, k_steps = M


def test_xla_layout_and_lazy_binding():
    from brl_b200 import _lib
    L = _lib.load()
    # keys, deal_table, pool, env_models, range offsets: operands; scratch; cum_return; sums in place; status; 2 x 6 Table_info
    assert L.brl_xla_layout(b"brl_duplicate_match") == b"iiiiisoxooooooooooooo"
    assert "brl_duplicate_match" in _lib.OPS and "brl_duplicate_match" in _lib.LAZY_OPS
    assert "brl_duplicate_match_xla" in _lib.XLA_LEGACY
    for name in ("brl_duplicate_match_scratch_bytes", "brl_duplicate_match_graph_builds"):
        assert name in _lib.MISC
        getattr(L, name)


def test_scratch_size_query():
    from brl_b200 import ops
    assert ops.duplicate_match_scratch_bytes(0, 2) == 0 and ops.duplicate_match_scratch_bytes(10, 0) == 0
    for n, M in ((1, 2), (100, 2), (4173, 2), (65536, 2), (1000, 17)):
        got = ops.duplicate_match_scratch_bytes(n, M)
        # at least the grouped forward's scratch and the env state, observation and mask; every piece 256-byte aligned
        assert got % 256 == 0
        assert got >= ops.policy_grouped_scratch_bytes(n, M) + n * (80 + 960 + 38)
    assert ops.duplicate_match_scratch_bytes(1000, 17) > ops.duplicate_match_scratch_bytes(1000, 2)
    assert ops.duplicate_match_scratch_bytes(2000, 2) > ops.duplicate_match_scratch_bytes(1000, 2)


def test_op_validates_its_arguments_without_a_gpu():
    from brl_b200 import _lib
    L = _lib.load()
    fn = _bind(L)

    def call(bufs, p, size=None):
        arr = (ctypes.c_void_p * 21)(*bufs)
        return fn(None, arr, ctypes.byref(p), ctypes.sizeof(p) if size is None else size)

    null = [None] * 21
    fake = [4096] * 9 + [None] * 12   # aligned, never dereferenced: each check below fails first
    assert call(null, _params(100, 2), 12) == -1 and b"BrlParams" in L.brl_last_error()
    # an empty batch is a no-op with NULL buffers
    assert call(null, _params(0, 2)) == 0
    assert call(null, _params(0, 5)) == 0
    # the pool's model count
    assert call(fake, _params(100, 0)) == -1 and b"model count" in L.brl_last_error()
    # without env_models the pool holds exactly two nets
    no_models = list(fake)
    no_models[3] = None
    assert call(no_models, _params(100, 3)) == -1 and b"2 nets" in L.brl_last_error()
    # the range count must come with the range offsets, and only with them
    no_ranges = list(fake)
    no_ranges[4] = None
    assert call(no_ranges, _params(100, 3, P=4)) == -1 and b"range" in L.brl_last_error()
    assert call(fake, _params(100, 3, P=0)) == -1 and b"range" in L.brl_last_error()
    assert call(fake, _params(100, 3, P=2, n_deals=0)) == -1 and b"n_deals" in L.brl_last_error()
    assert call(fake, _params(100, 3, P=2, flags=_lib.F_SAMPLE)) == -1 and b"sampling" in L.brl_last_error()
    # required buffers
    for k, name in ((0, b"keys"), (2, b"pool"), (5, b"scratch"), (6, b"cum_return"), (7, b"sums"), (8, b"status")):
        bufs = list(fake)
        bufs[k] = None
        assert call(bufs, _params(100, 3, P=2)) == -2 and name in L.brl_last_error(), name
    # the Table_info outputs come all twelve or not at all
    some = list(fake)
    some[9] = 4096
    assert call(some, _params(100, 3, P=2)) == -2 and b"Table_info" in L.brl_last_error()


def test_python_wrapper_checks_shapes_and_scratch_before_touching_the_device():
    from brl_b200 import _lib, ops
    n = 64
    keys, table = torch.zeros(n, dtype=torch.int64), torch.zeros((10, 48), dtype=torch.uint8)
    cum, status = torch.zeros(n), torch.zeros(1, dtype=torch.int32)
    pool2 = torch.zeros((2, ops.mlp_pool_stride()), dtype=torch.uint8)
    pool3 = torch.zeros((3, ops.mlp_pool_stride()), dtype=torch.uint8)
    sums = torch.zeros(8, dtype=torch.float64)
    small = torch.zeros(ops.duplicate_match_scratch_bytes(n, 2) - 1, dtype=torch.uint8)
    with pytest.raises(_lib.BrlError, match="2 nets"):
        ops.duplicate_match(keys, table, pool3, small, cum, sums, status)
    with pytest.raises(_lib.BrlError, match="scratch too small"):
        ops.duplicate_match(keys, table, pool2, small, cum, sums, status)
    with pytest.raises(_lib.BrlError, match="range_offsets"):
        ops.duplicate_match(keys, table, pool2, small, cum, torch.zeros((3, 8), dtype=torch.float64), status,
                            range_offsets=torch.zeros(3, dtype=torch.int64))
    with pytest.raises(_lib.BrlError, match="env_models"):
        ops.duplicate_match(keys, table, pool3, small, cum, sums, status, env_models=torch.zeros((n, 3), dtype=torch.int32))


def test_duplicate_eval_script_arguments():
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import duplicate_eval
    cfg = duplicate_eval.parse_args(["team1_model_path=a.pkl", "team2_model_path=b.pkl", "team1_activation=relu",
                                     "num_eval_envs=250"])
    assert cfg["team1_model_path"] == "a.pkl" and cfg["team2_model_path"] == "b.pkl" and cfg["num_eval_envs"] == 250
    assert cfg["team2_activation"] == "relu" and cfg["team1_model_type"] == "DeepMind"
    assert cfg["eval_dds"] == "dds_results/test_000.npy"
    for bad in (["bogus=1", "team1_model_path=a", "team2_model_path=b"], ["team1_model_path=a"],
                ["team1_model_path=a", "team2_model_path=b", "team2_activation=tanh"],
                ["team1_model_path=a", "team2_model_path=b", "num_eval_envs=0"]):
        with pytest.raises(SystemExit):
            duplicate_eval.parse_args(bad)
