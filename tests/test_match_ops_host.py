"""CPU: the argument checks of the three device-match ops (brl_duplicate_match, brl_evaluate_match, brl_call_values), called
through _lib.call with made-up 4096-aligned addresses that are never dereferenced.  Every case has exactly one defect, and a
check rejects it before any CUDA call.  Each case asserts the return code and, for a buffer, that the message names it."""
import re

import pytest

from brl_b200 import _lib

A = 4096
OPAQUE, BUFFER = -1, -2
DUP, SINGLE, SIMPLE = _lib.EVAL_MATCH_DUPLICATE, _lib.EVAL_MATCH_SINGLE, _lib.EVAL_MATCH_SIMPLE
TABLE_INFO = [f"table_{t}.{f}" for t in "ab" for f in ("terminated", "rewards", "last_bid", "last_bidder", "call_x", "call_xx")]
NAMES = {
    "brl_duplicate_match": ["keys", "deal_table", "pool", "env_models", "range offsets", "scratch", "cum_return", "sums",
                            "status"] + TABLE_INFO + ["system histogram [21]"],
    "brl_evaluate_match": ["keys", "deal_table", "pool", "scratch", "cum_return", "acc", "sums", "status"] + TABLE_INFO +
                          ["final state", "observation", "mask", "rewards", "terminated", "current_player"],
    "brl_call_values": ["keys", "deal_table", "pool", "env_models", "rewards_a", "rewards_b", "scratch", "gain_sums",
                        "regret_sums", "mismatch", "status", "count", "env", "table", "player", "net", "context", "played", "r",
                        "obs", "gain"],
}


def _params(n=100, *, n_deals=100, flags=0, step=0, k_steps=0, seed=0):
    return _lib.BrlParams(n, 0, 0, seed, n_deals, flags, step, k_steps, -1.0, 1.0, 0.0, 0.0)


# op -> (buffers given, params) of a call that passes every check; each case below changes one thing
def _dup():  # env_models [n, 2] and two ranges
    return ["keys", "deal_table", "pool", "env_models", "range offsets", "scratch", "cum_return", "sums", "status"], \
        _params(k_steps=3, step=2)


def _eval(mode=DUP):
    return NAMES["brl_evaluate_match"][:8], _params(flags=_lib.f_eval_match(mode))


def _cv():
    return NAMES["brl_call_values"][:11], _params(k_steps=2, seed=16)


def _call(op, given, params, misalign=None, by=0):
    buffers = [A if name in given else None for name in NAMES[op]]
    if misalign is not None:
        buffers[NAMES[op].index(misalign)] = A + by
    _lib.call(op, 0, buffers, params)


def _fails(rc, pattern, op, *args, **kw):
    with pytest.raises(_lib.BrlError, match=rf"^{op} failed \({rc}\): {op}: .*{pattern}"):
        _call(op, *args, **kw)


def _without(given, name):
    return [g for g in given if g != name]


@pytest.mark.parametrize("op,flags", [("brl_duplicate_match", 0), ("brl_call_values", 0)] +
                         [("brl_evaluate_match", _lib.f_eval_match(m)) for m in (0, DUP, SINGLE, SIMPLE)])
def test_empty_batch_is_a_no_op(op, flags):
    _call(op, [], _params(0, flags=flags))


REQUIRED = ([("brl_duplicate_match", _dup, b) for b in ("keys", "deal_table", "pool", "scratch", "cum_return", "sums", "status")] +
            [("brl_evaluate_match", _eval, b) for b in NAMES["brl_evaluate_match"][:8]] +
            [("brl_call_values", _cv, b) for b in NAMES["brl_call_values"][:11]])


@pytest.mark.parametrize("op,base,buf", REQUIRED)
def test_a_null_required_buffer_is_named(op, base, buf):
    given, p = base()
    _fails(BUFFER, re.escape(buf), op, _without(given, buf), p)


# (op, base, extra buffers given, buffer, its alignment)
ALIGNED = ([("brl_duplicate_match", _dup, [], b, a) for b, a in
            (("keys", 16), ("deal_table", 16), ("pool", 16), ("env_models", 8), ("range offsets", 8), ("scratch", 16),
             ("cum_return", 4), ("sums", 8), ("status", 4), ("system histogram [21]", 4))] +
           [("brl_duplicate_match", _dup, TABLE_INFO, b, 16) for b in ("table_a.rewards", "table_b.rewards")] +
           [("brl_evaluate_match", _eval, [], b, a) for b, a in
            (("keys", 16), ("deal_table", 16), ("pool", 16), ("scratch", 16), ("cum_return", 4), ("acc", 4), ("sums", 8),
             ("status", 4))] +
           [("brl_evaluate_match", _eval, TABLE_INFO, b, 16) for b in ("table_a.rewards", "table_b.rewards")] +
           [("brl_evaluate_match", lambda: _eval(SINGLE), NAMES["brl_evaluate_match"][20:], b, a) for b, a in
            (("final state", 16), ("observation", 16), ("mask", 2), ("rewards", 16))] +
           [("brl_call_values", _cv, [], b, a) for b, a in
            (("keys", 16), ("pool", 16), ("env_models", 16), ("rewards_a", 16), ("rewards_b", 16), ("scratch", 16),
             ("gain_sums", 8), ("regret_sums", 8), ("mismatch", 8), ("status", 4))] +
           [("brl_call_values", _cv, NAMES["brl_call_values"][11:19], b, a) for b, a in
            [("count", 8)] + [(r, 4) for r in ("env", "table", "player", "net", "context", "played", "r")]] +
           [("brl_call_values", _cv, NAMES["brl_call_values"][11:], b, a) for b, a in (("obs", 16), ("gain", 4))])


@pytest.mark.parametrize("op,base,extra,buf,align", ALIGNED, ids=[f"{c[0]}-{c[3]}" for c in ALIGNED])
def test_a_misaligned_buffer_is_named(op, base, extra, buf, align):
    given, p = base()
    _fails(BUFFER, re.escape(buf), op, given + extra, p, misalign=buf, by=align // 2)


# (op, base, buffers given beyond the base's, message): a group given in part
GROUPS = [
    ("brl_duplicate_match", _dup, ["table_a.terminated"], "Table_info"),
    ("brl_duplicate_match", _dup, TABLE_INFO[:11], "Table_info"),
    ("brl_evaluate_match", _eval, ["table_b.call_xx"], "Table_info"),
    ("brl_evaluate_match", lambda: _eval(SINGLE), ["final state"], "final-state"),
    ("brl_evaluate_match", lambda: _eval(SINGLE), NAMES["brl_evaluate_match"][21:], "final-state"),
    ("brl_call_values", _cv, ["count"], "record"),
    ("brl_call_values", _cv, NAMES["brl_call_values"][12:19], "record"),
    ("brl_call_values", _cv, NAMES["brl_call_values"][11:20], "training-example"),
    ("brl_call_values", _cv, NAMES["brl_call_values"][11:19] + ["gain"], "training-example"),
    ("brl_call_values", _cv, ["obs", "gain"], "record buffers"),
]


@pytest.mark.parametrize("op,base,extra,message", GROUPS)
def test_all_or_none_groups(op, base, extra, message):
    given, p = base()
    _fails(BUFFER, message, op, given + extra, p)


def _opaque_cases():
    dup, _ = _dup()
    ev, _ = _eval()
    cv, _ = _cv()
    no_models = _without(dup, "env_models")
    no_ranges = _without(dup, "range offsets")
    flags = _lib.f_eval_match(DUP)
    return [
        ("brl_duplicate_match", dup, _params(k_steps=0, step=2), "model count"),
        ("brl_duplicate_match", no_models, _params(k_steps=3, step=2), "2 nets"),
        ("brl_duplicate_match", no_models, _params(k_steps=2, step=2, flags=_lib.F_PLAYER_MODELS), "BRL_F_PLAYER_MODELS"),
        ("brl_duplicate_match", no_ranges, _params(k_steps=3, step=2), "range count"),
        ("brl_duplicate_match", dup, _params(k_steps=3, step=0), "range count"),
        ("brl_duplicate_match", dup, _params(1 << 30, k_steps=3, step=2), "n_envs"),
        ("brl_duplicate_match", dup, _params(k_steps=3, step=2, n_deals=0), "n_deals"),
        ("brl_duplicate_match", dup, _params(k_steps=3, step=2, flags=_lib.F_SAMPLE), "sampling"),
        ("brl_evaluate_match", ev, _params(), "mode"),
        ("brl_evaluate_match", ev, _params(flags=_lib.f_eval_match(SIMPLE) | _lib.F_EVAL_FREE_RUN), "FREE_RUN"),
        ("brl_evaluate_match", ev, _params(flags=flags | _lib.F_EVAL_PARTNER, k_steps=2), "BRL_F_EVAL_PARTNER"),
        ("brl_evaluate_match", ev, _params(1 << 30, flags=flags), "n_envs"),
        ("brl_evaluate_match", ev, _params(flags=flags, n_deals=0), "n_deals"),
        ("brl_evaluate_match", ev, _params(flags=flags | _lib.F_SAMPLE), "sampling"),
        ("brl_call_values", cv, _params(k_steps=0, seed=16), "model count"),
        ("brl_call_values", cv, _params(1 << 30, k_steps=2, seed=16), "n_envs"),
        ("brl_call_values", cv, _params(k_steps=2, seed=16, n_deals=0), "n_deals"),
        ("brl_call_values", cv, _params(k_steps=2, seed=16, flags=_lib.F_SAMPLE), "sampling"),
        ("brl_call_values", cv, _params(k_steps=2, seed=(1 << 64) - 1), "record capacity"),
    ]


OPAQUE_CASES = _opaque_cases()


@pytest.mark.parametrize("op,given,p,message", OPAQUE_CASES, ids=[f"{c[0]}-{c[3]}-{k}" for k, c in enumerate(OPAQUE_CASES)])
def test_opaque_checks(op, given, p, message):
    rc = BUFFER if message == "BRL_F_PLAYER_MODELS" else OPAQUE   # a missing buffer the flag needs
    _fails(rc, re.escape(message), op, given, p)
