"""CPU: counterfactual call values (DESIGN.md f16) -- gains and regret of hand-built decisions (tests/call_values_ref.py),
the reference reduction against hand sums, the report's statistics on a hand-made sums array, the op's registration and
XLA layout, the wrappers' and the op's argument checks, and the script's arguments."""
import ctypes
import math

import numpy as np
import pytest
import torch

from tests import call_values_ref as R

NAN = float("nan")


def _r(values):
    """r[38] with the given calls legal: {call: points}, NaN elsewhere"""
    r = np.full(38, np.nan, np.float32)
    for a, v in values.items():
        r[a] = v
    return r


def test_imp_matches_the_golden_table():
    import os
    table = np.load(os.path.join(os.path.dirname(__file__), "golden", "imp_table.npy"))
    diffs = np.arange(-5000, 5001, 10)
    if table.ndim == 1 and len(table) == len(diffs):
        assert [R.imp(float(d)) for d in diffs] == list(table)
    for d, want in ((0, 0), (19, 0), (20, 1), (-20, -1), (49, 1), (50, 2), (3999, 23), (4000, 24), (-7600, -24)):
        assert R.imp(d) == want, d


def test_gain_on_both_tables_and_teams():
    # table A: team 1 made 420, table B: team 1 (defending) lost 420 -> the board is a push
    R_a, R_b = 420.0, -420.0
    r = _r({0: 420.0, 3: 170.0, 30: -100.0})
    g = R.gains(r, R_a, R_b, table=0, player=0)
    assert g[0] == 0                                   # the played call (Pass, the base game) gains nothing
    assert g[3] == R.imp(170 - 420) == -6              # a partscore instead of the game: -6 for team 1
    assert g[30] == R.imp(-100 - 420) == -11
    assert g[1] is None and g[37] is None              # illegal: no branch
    # the same decision by team 2 (player 2): the sign flips
    assert R.gains(r, R_a, R_b, table=0, player=2)[3] == 6
    # table B: R_A is the other table
    gb = R.gains(_r({0: -420.0, 5: -50.0}), R_a, R_b, table=1, player=3)
    assert gb[0] == 0 and gb[5] == -(R.imp(420 - 50) - 0) == -9
    assert R.regret(gb) == 0 and R.regret(R.gains(r, R_a, R_b, table=0, player=2)) == 11


def test_gain_at_the_imp_table_edges():
    # base 0; a branch moving the board by exactly a threshold gains that threshold's IMPs, one point less does not
    for t, k in ((20, 1), (50, 2), (4000, 24)):
        g = R.gains(_r({0: 0.0, 3: float(t), 4: float(t - 1)}), 0.0, 0.0, table=0, player=1)
        assert g[3] == k and g[4] == k - 1
    # the largest swing: -24 at the base to +24 -> 48
    g = R.gains(_r({0: -4000.0, 9: 4000.0}), -4000.0, 0.0, table=0, player=0)
    assert g[9] == 48 and R.regret(g) == 48


def test_single_legal_call_after_7nt_redoubled():
    # after 7NT XX only Pass is legal: one branch, the played one, gain 0 and regret 0
    g = R.gains(_r({0: 2980.0}), 2980.0, -2980.0, table=0, player=2)
    assert [x for x in g if x is not None] == [0] and R.regret(g) == 0


def test_reduction_equals_hand_sums():
    rec = dict(env=np.array([0, 0, 1]), table=np.array([0, 1, 0]), player=np.array([0, 2, 1]), net=np.array([0, 0, 1]),
               context=np.array([0, 74, 0]), played=np.array([0, 3, 0]),
               r=np.stack([_r({0: 420.0, 3: 170.0}), _r({0: -450.0, 3: -420.0, 4: -400.0}), _r({0: 50.0, 3: 110.0})]))
    R_a, R_b = np.array([420.0, 50.0]), np.array([-420.0, 0.0])
    gain, reg, mismatch = R.reduce_records(rec, R_a, R_b, 2)
    # decision 0: net 0, OPEN(0), Pass played: g = {Pass: 0, 1C: -6}
    assert tuple(gain[0, 0, 0, 0]) == (1, 0, 0, 0) and tuple(gain[0, 0, 0, 3]) == (1, -6, 36, 0)
    # decision 1: table B, player 2 (team 2), 1C played (r = -420 = R_B): Pass would gain 1, 1D lose 1
    g1 = R.gains(rec["r"][1], 420.0, -420.0, 1, 2)
    assert g1[3] == 0 and g1[0] == -R.imp(420 - 450) == 1 and g1[4] == -R.imp(420 - 400) == -1
    assert tuple(gain[0, 74, 3, 0]) == (1, 1, 1, 1) and tuple(gain[0, 74, 3, 4]) == (1, -1, 1, 0)
    # decision 2: net 1, R_T = 50 (2 IMPs on the board), 1C would make 110 (3 IMPs): +1
    assert tuple(gain[1, 0, 0, 3]) == (1, 1, 1, 1) and tuple(reg[1, 0]) == (1, 1, 1, 1)
    assert tuple(reg[0, 0]) == (1, 0, 0, 0) and tuple(reg[0, 74]) == (1, 1, 1, 1)
    assert list(mismatch) == [0, 0]
    rec["r"][2][0] = 60.0                                    # the played branch differs from the base result
    assert list(R.reduce_records(rec, R_a, R_b, 2)[2]) == [0, 1]


def test_report_statistics_of_hand_made_sums():
    from brl_b200 import call_values, system
    from brl_b200.board_log import ACTION_STR
    gain = np.zeros((75, 38, 38, 4), np.int64)
    regret = np.zeros((75, 4), np.int64)
    xs = np.array([3, 5, 0, 6, 3, 1])                       # OPEN(0): Pass played, 1NT instead
    gain[0, 0, 3 + 4] = (len(xs), xs.sum(), (xs * xs).sum(), (xs > 0).sum())
    gain[0, 0, 0] = (len(xs), 0, 0, 0)
    gain[5, 3, 4] = (2, 10, 50, 2)                           # too few decisions
    regret[0] = (len(xs), xs.sum(), (xs * xs).sum(), (xs > 0).sum())
    regret[74] = (4, 0, 0, 0)
    v = call_values.CallValues(gain, regret, 0)
    assert v.decisions == 10 and v.mean_regret() == pytest.approx(18 / 10)
    top = v.top_deviations(k=5, min_count=3)
    assert len(top) == 1 and top[0]["played"] == ACTION_STR[0] and top[0]["instead"] == ACTION_STR[7]
    assert top[0]["context"] == system.context_name(0)
    assert top[0]["mean"] == pytest.approx(3.0) and top[0]["total_imps"] == 18
    assert top[0]["se"] == pytest.approx(np.std(xs, ddof=1) / math.sqrt(len(xs)))
    table = v.regret_table()
    assert [t["decisions"] for t in table] == [6, 4] and table[0]["share_positive"] == pytest.approx(5 / 6)
    doubled = regret.copy()
    doubled[:, 1:3] *= 2
    worse = call_values.CallValues(gain, doubled, 0)
    cmp = call_values.compare(v, worse)
    assert cmp["mean_regret_change"] == pytest.approx(18 / 10)
    res = dict(gain_sums=gain[None], regret_sums=regret[None], mismatch=np.zeros(1, np.int64))
    assert call_values.from_sums(res)[0].decisions == 10
    assert v.summary(5, 3)["top_deviations"] == top


def test_op_is_registered_with_its_xla_layout():
    from brl_b200 import _lib
    L = _lib.load()
    assert "brl_call_values" in _lib.OPS and "brl_call_values" in _lib.LAZY_OPS and "brl_call_values_xla" in _lib.XLA_LEGACY
    L.brl_xla_layout.restype = ctypes.c_char_p
    assert L.brl_xla_layout(b"brl_call_values") == b"iiiiiisoooooooooooo"
    assert "brl_call_values_scratch_bytes" in _lib.MISC


def test_wrappers_check_their_arguments_before_any_device_work():
    from brl_b200 import _lib, ops
    n, M = 4, 2
    keys, pool = torch.zeros(n, dtype=torch.int64), torch.zeros((M, ops.mlp_pool_stride()), dtype=torch.uint8)
    table = torch.zeros((100, 48), dtype=torch.uint8)
    em, ra, rb = torch.zeros((n, 2), dtype=torch.int32), torch.zeros((n, 4)), torch.zeros((n, 4))
    gain = torch.zeros((M,) + ops.CALL_GAIN_SHAPE, dtype=torch.int64)
    reg = torch.zeros((M,) + ops.CALL_REGRET_SHAPE, dtype=torch.int64)
    mm, st, scratch = torch.zeros(M, dtype=torch.int64), torch.zeros(1, dtype=torch.int32), torch.zeros(16, dtype=torch.uint8)
    args = [keys, table, pool, em, ra, rb, scratch, gain, reg, mm, st]

    def bad(k, v, match):
        a = list(args)
        a[k] = v
        with pytest.raises(_lib.BrlError, match=match):
            ops.call_values(*a)

    bad(0, keys.int(), "keys")
    bad(2, pool[:, :8], "pool")
    bad(3, torch.zeros((n, 3), dtype=torch.int32), "env_models")
    bad(4, torch.zeros((n, 4), dtype=torch.float64), "rewards_a")
    bad(5, torch.zeros((n + 1, 4)), "rewards_b")
    bad(1, table[:, :40], "deal table")
    bad(7, gain[:1], "gain_sums")
    bad(8, reg.int(), "regret_sums")
    bad(9, mm[:1], "mismatch")
    bad(10, st.long(), "status")
    bad(6, scratch, "scratch too small")
    a = list(args)
    a[6] = torch.zeros(ops.call_values_scratch_bytes(n, M), dtype=torch.uint8)
    with pytest.raises(_lib.BrlError, match="sampling"):
        ops.call_values(*a, tune=_lib.F_SAMPLE)
    with pytest.raises(_lib.BrlError, match="CUDA"):          # every shape right: the first thing left is the device
        ops.call_values(*a)


def test_the_op_checks_its_buffers():
    from brl_b200 import _lib
    L = _lib.load()
    fn = L.brl_call_values
    fn.restype, fn.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]
    p0 = _lib.BrlParams(0, 0, 0, 0, 100, 0, 0, 2, -1.0, 1.0, 0.0, 0.0)
    assert fn(None, (ctypes.c_void_p * 19)(), ctypes.byref(p0), ctypes.sizeof(p0)) == 0           # an empty batch: a no-op
    p = _lib.BrlParams(10, 0, 0, 0, 100, 0, 0, 2, -1.0, 1.0, 0.0, 0.0)
    names = ["keys", "deal_table", "pool", "env_models", "rewards_a", "rewards_b", "scratch", "gain_sums", "regret_sums",
             "mismatch", "status"]
    for k, name in enumerate(names):                                                             # a NULL required buffer
        b = [4096] * 11 + [None] * 8
        b[k] = None
        assert fn(None, (ctypes.c_void_p * 19)(*b), ctypes.byref(p), ctypes.sizeof(p)) == -2
        assert name.encode() in L.brl_last_error()
    b = [4096] * 11 + [4096] * 7 + [None]                                                         # records: all or none
    assert fn(None, (ctypes.c_void_p * 19)(*b), ctypes.byref(p), ctypes.sizeof(p)) == -2
    assert b"record" in L.brl_last_error()
    for bad in (_lib.BrlParams(10, 0, 0, 0, 100, 0, 0, 0, -1.0, 1.0, 0.0, 0.0),                  # M = 0
                _lib.BrlParams(10, 0, 0, 0, 100, _lib.F_SAMPLE, 0, 2, -1.0, 1.0, 0.0, 0.0),      # sampling
                _lib.BrlParams(10, 0, 0, 0, 0, 0, 0, 2, -1.0, 1.0, 0.0, 0.0)):                   # no deals
        assert fn(None, (ctypes.c_void_p * 19)(*([4096] * 11 + [None] * 8)), ctypes.byref(bad), ctypes.sizeof(bad)) == -1


def test_script_parses_its_arguments():
    import importlib
    script = importlib.import_module("scripts.call_values")
    cfg = script.parse_args(["nets=a.pkl,b.pkl", "num_eval_envs=64", "opponent=1", "top=5"])
    assert script.net_paths(cfg) == ["a.pkl", "b.pkl"] and cfg["num_eval_envs"] == 64 and cfg["opponent"] == 1
    assert cfg["top"] == 5 and cfg["min_count"] == 30
    with pytest.raises(SystemExit):
        script.parse_args([])
    with pytest.raises(SystemExit):
        script.parse_args(["nope=1", "nets=a.pkl"])


def test_chunk_bytes_follow_the_buffer_list():
    from brl_b200 import evaluation as ev, ops
    n, M = 1000, 2
    base = ev.call_values_bytes(n, M)
    assert base > ops.call_values_scratch_bytes(n, M) + ops.duplicate_match_scratch_bytes(n, M)
    assert ev.call_values_bytes(n, M, 10) - base == 10 * (6 * 4 + 38 * 4) + 8
