"""CPU: the argument checks of the loss-head ops that take a BrlSlParams (brl_sl_grad / brl_sl_eval, brl_cv_grad /
brl_cv_eval), called through _lib.call.  Each check runs before any CUDA call, so no device is needed.  No case here
passes every check: the made-up addresses below must never reach a launch.  Every case but the ones about `acc` also
leaves `acc` (the last buffer) NULL, so the buffer under test must be the first one reported."""
import ctypes

import pytest

from brl_b200 import _lib

# name -> (buffers in order, the 16-byte-aligned ones); gain (CV) must be 4-byte aligned
OPS = {
    "brl_sl_grad": (["obs", "blob", "scratch", "mask", "label", "grads", "stats", "acc"], {"obs", "blob", "scratch", "grads", "acc"}),
    "brl_sl_eval": (["obs", "blob", "scratch", "mask", "label", "stats", "acc"], {"obs", "blob", "scratch", "acc"}),
    "brl_cv_grad": (["obs", "blob", "scratch", "gain", "grads", "stats", "acc"], {"obs", "blob", "scratch", "grads", "acc"}),
    "brl_cv_eval": (["obs", "blob", "scratch", "gain", "stats", "acc"], {"obs", "blob", "scratch", "acc"}),
}
CASES = [(op, buf) for op, (names, _) in OPS.items() for buf in names]
MISALIGNED = [(op, buf) for op, (_, aligned) in OPS.items() for buf in sorted(aligned)]


def _buffers(op, null=None, misalign=None, by=16):
    """made-up 16-byte-aligned addresses, one of them NULL or moved by `by` bytes, plus a later defect that fails too"""
    names = OPS[op][0]
    addr = {n: 0x10000 * (k + 1) for k, n in enumerate(names)}
    if null is not None:
        addr[null] = None
    if misalign is not None:
        addr[misalign] += by
    if "acc" not in (null, misalign):
        addr["acc"] = None
    elif "gain" in addr:
        addr["gain"] += 2
    return [addr[n] for n in names]


def _fails(op, buffers, params, rc, message):
    with pytest.raises(_lib.BrlError, match=rf"^{op} failed \({rc}\): {message}"):
        _lib.call(op, 0, buffers, params)


@pytest.mark.parametrize("op", sorted(OPS))
def test_empty_batch_is_a_no_op(op):
    _lib.call(op, 0, [None] * len(OPS[op][0]), _lib.BrlSlParams(0, 0.0, 0))


@pytest.mark.parametrize("op", sorted(OPS))
def test_opaque_must_be_one_sl_params(op):
    class Short(ctypes.Structure):
        _fields_ = [("batch", ctypes.c_int64)]
    _fails(op, _buffers(op, null="obs"), Short(4), -1, rf"{op}: opaque must be one BrlSlParams")


@pytest.mark.parametrize("batch", [-1, (1 << 24) + 1])
@pytest.mark.parametrize("op", sorted(OPS))
def test_batch_out_of_range(op, batch):
    _fails(op, _buffers(op, null="obs"), _lib.BrlSlParams(batch, 0.0, 0), -1, rf"{op}: batch must be in \[0, 2\^24\]")


@pytest.mark.parametrize("op,buf", CASES)
def test_a_null_buffer_is_named(op, buf):
    _fails(op, _buffers(op, null=buf), _lib.BrlSlParams(4, 0.0, 0), -2, rf"{op}: buffer '{buf}' is NULL")


@pytest.mark.parametrize("op,buf", MISALIGNED)
def test_a_misaligned_buffer_is_named(op, buf):
    _fails(op, _buffers(op, misalign=buf, by=8), _lib.BrlSlParams(4, 0.0, 0), -2, rf"{op}: buffer '{buf}' is not 16-byte aligned")


@pytest.mark.parametrize("op", ["brl_cv_eval", "brl_cv_grad"])
def test_a_misaligned_gain_is_named(op):
    names = OPS[op][0]
    buffers = [0x10000 * (k + 1) for k in range(len(names))]
    buffers[names.index("gain")] += 2  # the only defect: the gain check follows the buffer checks, with no check after it
    _fails(op, buffers, _lib.BrlSlParams(4, 0.0, 0), -2, rf"{op}: gain is not 4-byte aligned")
