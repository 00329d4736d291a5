"""CPU: ops with a group of optional buffers report a broken group before they look at the optional buffers after it, so the
message names the first problem in buffer order (made-up addresses that are never dereferenced; no GPU needed)."""
import ctypes

from brl_b200 import _lib

BAD = 4096 + 1  # misaligned for every buffer that has an alignment rule


def _fn(L, name):
    fn = getattr(L, name)
    fn.restype, fn.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]
    return fn


def test_call_values_reports_the_record_group_before_the_examples():
    L = _lib.load()
    fn = _fn(L, "brl_call_values")
    p = _lib.BrlParams(10, 0, 0, 0, 100, 0, 0, 2, -1.0, 1.0, 0.0, 0.0)
    b = [4096] * 18 + [None] + [BAD, BAD]  # seven of the eight record buffers, misaligned examples
    assert fn(None, (ctypes.c_void_p * 21)(*b), ctypes.byref(p), ctypes.sizeof(p)) == -2
    assert b"record" in L.brl_last_error()
    b = [4096] * 11 + [None] * 8 + [BAD, BAD]  # the examples alone are then checked
    assert fn(None, (ctypes.c_void_p * 21)(*b), ctypes.byref(p), ctypes.sizeof(p)) == -2
    assert b"aligned" in L.brl_last_error()


def test_duplicate_match_reports_the_table_info_group_before_the_histogram():
    L = _lib.load()
    fn = _fn(L, "brl_duplicate_match")
    p = _lib.BrlParams(100, 0, 0, 0, 10, 0, 2, 3, -1.0, 1.0, 0.0, 0.0)
    b = [4096] * 10 + [None] * 11 + [BAD]  # one Table_info buffer of twelve, a misaligned histogram
    assert fn(None, (ctypes.c_void_p * 22)(*b), ctypes.byref(p), ctypes.sizeof(p)) == -2
    assert b"Table_info" in L.brl_last_error()


def test_hand_posterior_smc_reports_the_particle_group_before_the_trace():
    L = _lib.load()
    fn = _fn(L, "brl_hand_posterior_smc")
    p = _lib.BrlSmcParams(_lib.BrlParams(4, 0, 1024, 0, 10, 0, 64, 2, -1.0, 1.0, 1.0, 0.0), 0.5, 2, 40, 0)
    b = [4096 * (k + 1) for k in range(18)] + [None] * 2 + [BAD] * 5  # hands without logw / ell, a misaligned trace
    assert fn(None, (ctypes.c_void_p * 25)(*b), ctypes.byref(p), ctypes.sizeof(p)) == -2
    assert b"go together" in L.brl_last_error()
