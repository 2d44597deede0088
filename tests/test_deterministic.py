"""The deterministic-mode switch of the C ABI round-trips without touching CUDA (no GPU needed)."""


def test_deterministic_mode_round_trip():
    import d2d_ppo_b200
    from d2d_ppo_b200 import _lib
    lib = _lib.lib()
    before = lib.d2d_get_deterministic()
    assert before == 0                                       # off by default
    try:
        for mode in (True, False, True):
            d2d_ppo_b200.use_deterministic_algorithms(mode)
            assert d2d_ppo_b200.are_deterministic_algorithms_enabled() is mode
            assert lib.d2d_get_deterministic() == int(mode)
        assert lib.d2d_set_deterministic(7) == _lib.OK and lib.d2d_get_deterministic() == 1   # any non-zero is on
    finally:
        lib.d2d_set_deterministic(before)
    assert lib.d2d_get_deterministic() == before
