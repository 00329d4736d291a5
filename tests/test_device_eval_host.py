"""CPU: the host side of brl_evaluate_match (make_evaluate / make_simple_evaluate as one device-resident call) -- its XLA
layout, lazy binding, argument validation, scratch-size query, and the evaluators ppo.train builds."""
import ctypes
import os
import subprocess
import sys

import pytest
import torch

N_BUFFERS = 26


def _bind(L):
    fn = L.brl_evaluate_match
    fn.restype, fn.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]
    return fn


def _params(n, mode, n_deals=100, flags=0):
    from brl_b200 import _lib
    return _lib.BrlParams(n, 0, 0, 0, n_deals, _lib.f_eval_match(mode) | flags, 0, 0, -1.0, 1.0, 0.0, 0.0)


def test_xla_layout_and_lazy_binding():
    from brl_b200 import _lib
    L = _lib.load()
    # keys, deal_table, pool: operands; scratch; cum_return; acc; sums in place; status; 2 x 6 Table_info; 6 final-state outputs
    assert L.brl_xla_layout(b"brl_evaluate_match") == b"iiisoox" + b"o" * 19
    assert "brl_evaluate_match" in _lib.OPS and "brl_evaluate_match" in _lib.LAZY_OPS
    assert "brl_evaluate_match_xla" in _lib.XLA_LEGACY
    assert "brl_evaluate_match_scratch_bytes" in _lib.MISC
    # load() leaves the lazy op unbound (checked in a fresh process: other tests call it): a process that never calls it
    # creates no extra ctypes objects
    code = ("from brl_b200 import _lib; L = _lib.load(); "
            "assert L.brl_evaluate_match.argtypes is None and L.brl_evaluate_match_xla.argtypes is None")
    subprocess.run([sys.executable, "-c", code], check=True, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def test_scratch_size_query():
    from brl_b200 import _lib, ops
    modes = (_lib.EVAL_MATCH_DUPLICATE, _lib.EVAL_MATCH_SINGLE, _lib.EVAL_MATCH_SIMPLE)
    for mode in modes:
        assert ops.evaluate_match_scratch_bytes(0, mode) == 0
    for bad in (0, 4, -1):
        assert ops.evaluate_match_scratch_bytes(100, bad) == 0
    for n in (1, 100, 4097, 10000):
        base = ops.duplicate_match_scratch_bytes(n, 2)   # the duplicate loop's pieces, then each mode's own
        dup, single, simple = (ops.evaluate_match_scratch_bytes(n, m) for m in modes)
        assert dup % 256 == 0 and single % 256 == 0 and simple % 256 == 0
        assert dup >= base + n * (38 * 4 + 4 * 4 + 2)           # logits, step_count / last_bid / last_bidder / pass_num, call_x/xx
        assert single >= dup + n * 16                            # the summed rewards
        assert base + n <= simple < dup                          # the initial player
    assert ops.evaluate_match_scratch_bytes(2000, 1) > ops.evaluate_match_scratch_bytes(1000, 1)


def test_op_validates_its_arguments_without_a_gpu():
    from brl_b200 import _lib
    L = _lib.load()
    fn = _bind(L)
    DUP, SINGLE, SIMPLE = _lib.EVAL_MATCH_DUPLICATE, _lib.EVAL_MATCH_SINGLE, _lib.EVAL_MATCH_SIMPLE

    def call(bufs, p, size=None):
        arr = (ctypes.c_void_p * N_BUFFERS)(*bufs)
        return fn(None, arr, ctypes.byref(p), ctypes.sizeof(p) if size is None else size)

    def err():
        return L.brl_last_error()

    null = [None] * N_BUFFERS
    fake = [4096] * 8 + [None] * 18   # aligned, never dereferenced: each check below fails first
    assert call(null, _params(100, DUP), 12) == -1 and b"BrlParams" in err()
    # an empty batch is a no-op with NULL buffers, whatever the mode
    for mode in (0, DUP, SINGLE, SIMPLE):
        assert call(null, _params(0, mode)) == 0
    # the mode
    assert call(fake, _params(100, 0)) == -1 and b"mode" in err()
    assert call(fake, _params(100, SIMPLE, flags=_lib.F_EVAL_FREE_RUN)) == -1 and b"FREE_RUN" in err()
    assert call(fake, _params(100, DUP, n_deals=0)) == -1 and b"n_deals" in err()
    assert call(fake, _params(100, DUP, flags=_lib.F_SAMPLE)) == -1 and b"sampling" in err()
    # required buffers
    for k, name in ((0, b"keys"), (1, b"deal_table"), (2, b"pool"), (3, b"scratch"), (4, b"cum_return"), (5, b"acc"),
                    (6, b"sums"), (7, b"status")):
        bufs = list(fake)
        bufs[k] = None
        assert call(bufs, _params(100, DUP)) == -2 and name in err(), name
    # simple evaluate reads no acc / sums
    simple = list(fake)
    simple[5] = simple[6] = None
    assert call(simple, _params(0, SIMPLE)) == 0
    # misalignment
    for k, off, name in ((0, 8, b"keys"), (4, 2, b"cum_return"), (6, 4, b"sums"), (7, 1, b"status")):
        bufs = list(fake)
        bufs[k] = 4096 + off
        assert call(bufs, _params(100, DUP)) == -2 and name in err(), name
    # the Table_info outputs (duplicate) come all twelve or not at all, with 16-byte aligned rewards
    some = list(fake)
    some[8] = 4096
    assert call(some, _params(100, DUP)) == -2 and b"Table_info" in err()
    tables = list(fake[:8]) + [4096] * 12 + [None] * 6
    tables[9] = 4096 + 4
    assert call(tables, _params(100, DUP)) == -2 and b"16-byte" in err()
    # the final state (single table) likewise: all six or none, aligned
    some = list(fake)
    some[20] = 4096
    assert call(some, _params(100, SINGLE)) == -2 and b"final-state" in err()
    finals = list(fake[:8]) + [None] * 12 + [4096] * 6
    finals[21] = 4096 + 2
    assert call(finals, _params(100, SINGLE)) == -2 and b"aligned" in err()


def test_python_wrapper_checks_shapes_and_scratch_before_touching_the_device():
    from brl_b200 import _lib, ops
    n = 64
    keys, table = torch.zeros(n, dtype=torch.int64), torch.zeros((10, 48), dtype=torch.uint8)
    cum, status = torch.zeros(n), torch.zeros(1, dtype=torch.int32)
    pool2 = torch.zeros((2, ops.mlp_pool_stride()), dtype=torch.uint8)
    pool3 = torch.zeros((3, ops.mlp_pool_stride()), dtype=torch.uint8)
    acc, sums = torch.zeros((n, _lib.EVAL_ACC_COLS)), torch.zeros(_lib.load().brl_eval_num_sums(), dtype=torch.float64)
    small = torch.zeros(ops.evaluate_match_scratch_bytes(n, _lib.EVAL_MATCH_DUPLICATE) - 1, dtype=torch.uint8)
    with pytest.raises(_lib.BrlError, match="unknown mode"):
        ops.evaluate_match(keys, table, pool2, small, cum, status, mode=0, acc=acc, sums=sums)
    with pytest.raises(_lib.BrlError, match="free_run"):
        ops.evaluate_match(keys, table, pool2, small, cum, status, mode=_lib.EVAL_MATCH_SIMPLE, free_run=True)
    with pytest.raises(_lib.BrlError, match="pool"):
        ops.evaluate_match(keys, table, pool3, small, cum, status, mode=_lib.EVAL_MATCH_DUPLICATE, acc=acc, sums=sums)
    with pytest.raises(_lib.BrlError, match="acc"):
        ops.evaluate_match(keys, table, pool2, small, cum, status, mode=_lib.EVAL_MATCH_DUPLICATE, sums=sums)
    with pytest.raises(_lib.BrlError, match="scratch too small"):
        ops.evaluate_match(keys, table, pool2, small, cum, status, mode=_lib.EVAL_MATCH_DUPLICATE, acc=acc, sums=sums)


def test_ppo_train_builds_the_device_evaluators(monkeypatch):
    """ppo.train's evaluators: the three device loops, whatever the config"""
    from brl_b200 import ppo
    made = []
    for name in ("make_device_simple_evaluate", "make_device_duplicate_evaluate", "make_device_evaluate"):
        monkeypatch.setattr(ppo, name, lambda *a, _name=name, **kw: made.append(_name) or _name)
    cfg = ppo.default_config()
    assert ppo.make_evaluators(cfg, None, None) == ("make_device_simple_evaluate", "make_device_duplicate_evaluate",
                                                    "make_device_evaluate")
    assert made == ["make_device_simple_evaluate", "make_device_duplicate_evaluate", "make_device_evaluate"]
