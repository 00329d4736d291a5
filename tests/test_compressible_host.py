"""CPU: brl_alloc_compressible rounds every request up to the allocation granularity (brl_round_up_granularity)."""


def test_round_up_to_granularity():
    from brl_b200 import _lib
    L = _lib.load()
    g = 2 << 20
    cases = {1: g, g - 1: g, g: g, g + 1: 2 * g, 503_316_480: 503_316_480, 9_961_472: 10 * (1 << 20)}
    for b, want in cases.items():
        assert L.brl_round_up_granularity(b, g) == want, b
    assert L.brl_round_up_granularity(12345, 64 << 10) == 64 << 10
    assert L.brl_round_up_granularity((1 << 40) + 1, g) == (1 << 40) + g
    assert L.brl_round_up_granularity(777, 0) == 777
