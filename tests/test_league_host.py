"""CPU: the self-play league's host side -- checkpoint selection (workspace/eval_selfplay_league.py), the win/lose matrices,
argument validation of brl_model_rows / brl_policy_act_grouped / brl_match_stats_ranges and their size queries."""
import ctypes
import os

import numpy as np
import pytest


def _touch(d, names):
    for name in names:
        open(os.path.join(d, name), "wb").close()


def test_checkpoint_selection_follows_the_script(tmp_path):
    from brl_b200.evaluation import list_league_checkpoints
    run = tmp_path / "exp"
    run.mkdir()
    steps = [0, 50, 100, 150, 200, 300, 1000, 10000, 10100]
    _touch(run, [f"params-{s:08}.pkl" for s in steps])            # ppo.train's names
    _touch(run, [f"opt_state-{s:08}.pkl" for s in steps])         # never selected: no "params" in the name
    _touch(run, ["notes.txt", "model-sl.pkl"])
    got = list_league_checkpoints(str(tmp_path), "exp", skip_interval=100, max_step=10000)
    assert got == [f"params-{s:08}.pkl" for s in (0, 100, 200, 300, 1000, 10000)]
    assert list_league_checkpoints(str(tmp_path), "exp", skip_interval=50, max_step=150) == \
        [f"params-{s:08}.pkl" for s in (0, 50, 100, 150)]
    # unpadded names: the script sorts by name, not by step
    run2 = tmp_path / "raw"
    run2.mkdir()
    _touch(run2, ["params-200.pkl", "params-1000.pkl", "params-300.pkl"])
    assert list_league_checkpoints(str(tmp_path), "raw", 100, 10000) == ["params-1000.pkl", "params-200.pkl", "params-300.pkl"]
    _touch(run2, ["params.pkl"])
    with pytest.raises(ValueError, match="params.pkl"):
        list_league_checkpoints(str(tmp_path), "raw", 100, 10000)


def test_league_matrices_are_antisymmetric_with_sign_and_clip():
    from brl_b200.evaluation import league_matrices
    imps = {(0, 1): 2.5, (0, 2): -0.25, (0, 3): 0.0, (1, 2): -3.0, (1, 3): 0.75, (2, 3): 1.0}
    wl, dis, clip = league_matrices(4, imps)
    for m in (wl, dis, clip):
        assert np.array_equal(m, -m.T) and not np.diag(m).any()
    for (i, j), imp in imps.items():
        assert wl[j, i] == imp and wl[i, j] == -imp
        assert dis[j, i] == np.sign(imp) and dis[i, j] == -np.sign(imp)
        assert clip[j, i] == min(1.0, max(-1.0, imp))
    assert np.abs(clip).max() <= 1.0 and set(np.unique(dis)) <= {-1.0, 0.0, 1.0}
    assert dis[3, 0] == 0.0   # a tie stays 0, as in the script


def test_league_size_queries():
    from brl_b200 import _lib, ops
    L = _lib.load()
    stride = ops.mlp_pool_stride()
    assert stride == L.brl_mlp_packed_bytes() and stride % 256 == 0
    assert ops.model_rows_capacity(0, 5) == 0 and ops.model_rows_capacity(10, 0) == 0
    assert ops.model_rows_capacity(1, 1) == 256
    assert ops.model_rows_capacity(256, 1) == 256 and ops.model_rows_capacity(257, 1) == 512
    assert ops.model_rows_capacity(3, 17) == 3 * 256        # at most one group per env
    # the largest padded total: every non-empty group rounded up to 256 rows
    for n, m in ((1000, 3), (5050 * 100, 101), (129, 2)):
        cap = ops.model_rows_capacity(n, m)
        assert cap % 256 == 0 and cap >= n + min(n, m) * 255 - 255 and cap <= n + min(n, m) * 256
    assert ops.policy_grouped_scratch_bytes(1000, 3) == L.brl_mlp_rows_scratch_bytes(ops.model_rows_capacity(1000, 3))


def test_league_ops_validate_their_arguments_without_a_gpu():
    from brl_b200 import _lib
    L = _lib.load()
    for name in ("brl_model_rows", "brl_policy_act_grouped", "brl_match_stats_ranges"):
        fn = getattr(L, name)
        fn.restype, fn.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]

    def call(name, bufs, p, size=None):
        arr = (ctypes.c_void_p * 9)(*bufs)
        return getattr(L, name)(None, arr, ctypes.byref(p), ctypes.sizeof(p) if size is None else size)

    p = _lib.BrlParams(512, 0, 0, 0, 0, 0, 0, 3, 0.0, 0.0, 0.0, 0.0)   # n_envs, ..., k_steps = M
    null = [None] * 9
    fake = [4096] * 9   # aligned, never dereferenced: each check below fails first
    for name in ("brl_model_rows", "brl_policy_act_grouped", "brl_match_stats_ranges"):
        assert call(name, null, p, 12) == -1 and b"BrlParams" in L.brl_last_error()
        assert call(name, null, p) == -2 and b"NULL" in L.brl_last_error()
    # an empty batch is a no-op with NULL buffers
    p0 = _lib.BrlParams(0, 0, 0, 0, 0, 0, 0, 3, 0.0, 0.0, 0.0, 0.0)
    for name in ("brl_policy_act_grouped", "brl_match_stats_ranges"):
        assert call(name, null, p0) == 0
    bad = [4096, 4096, 4096, 4097, 4096, 4096, 4096, 4096, 4096]
    assert call("brl_policy_act_grouped", bad, p) == -2 and b"mask" in L.brl_last_error()
    # n_rows (buffer 8) points at offsets[M]: one int32, 4-byte aligned is enough
    assert call("brl_policy_act_grouped", fake[:8] + [None], p) == -2 and b"n_rows" in L.brl_last_error()
    assert call("brl_policy_act_grouped", fake[:8] + [4098], p) == -2 and b"n_rows" in L.brl_last_error()
    assert call("brl_policy_act_grouped", fake[:3] + [4097] + fake[4:8] + [4100], p) == -2 and b"mask" in L.brl_last_error()
    pk = _lib.BrlParams(512, 0, 0, 0, 0, 0, 0, 0, 0.0, 0.0, 0.0, 0.0)
    assert call("brl_policy_act_grouped", fake, pk) == -1 and b"model count" in L.brl_last_error()
    assert call("brl_model_rows", fake, pk) == -1 and b"model count" in L.brl_last_error()
    p300 = _lib.BrlParams(300, 0, 0, 0, 0, 0, 0, 3, 0.0, 0.0, 0.0, 0.0)
    assert call("brl_policy_act_grouped", fake, p300) == -1 and b"multiple of 256" in L.brl_last_error()
    ps = _lib.BrlParams(512, 0, 0, 0, 0, _lib.F_SAMPLE, 0, 3, 0.0, 0.0, 0.0, 0.0)
    assert call("brl_policy_act_grouped", fake, ps) == -1 and b"sampling" in L.brl_last_error()
    for name in ("brl_model_rows", "brl_policy_act_grouped", "brl_match_stats_ranges"):
        assert L.brl_xla_layout(name.encode()) is not None
    assert L.brl_xla_layout(b"brl_policy_act_grouped") == b"iisixiixi"


def test_league_ops_are_bound_lazily():
    """bench.py's process never creates their ctypes bindings (binding at load moved its rollout leg by 8 %)"""
    from brl_b200 import _lib
    for name in ("brl_model_rows", "brl_policy_act_grouped", "brl_match_stats_ranges"):
        assert name in _lib.OPS and name in _lib.LAZY_OPS


def test_selfplay_league_script_arguments():
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import selfplay_league
    cfg = selfplay_league.parse_args(["exp_name=run1", "num_eval_envs=50", "skip_interval=10", "max_step=200"])
    assert cfg["exp_name"] == "run1" and cfg["num_eval_envs"] == 50 and cfg["skip_interval"] == 10 and cfg["max_step"] == 200
    assert cfg["models_directory"] == "models" and cfg["activation"] == "relu"
    with pytest.raises(SystemExit):
        selfplay_league.parse_args(["bogus=1"])
