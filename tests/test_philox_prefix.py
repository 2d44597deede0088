"""The two-round split of Philox4x32-10 that comb_run_kernel uses (philox.cuh: philox_env_head, philox_call_head and
the philox overload that continues from them), restated in numpy and checked against oracle.philox_np.philox4x32_10
over random counters and keys, block words other than 0 included."""
import numpy as np

from oracle import philox_np as px

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
U32 = np.uint64(0xFFFFFFFF)


def _mul(m, x):
    p = np.uint64(m) * np.asarray(x, dtype=np.uint64)
    return p >> np.uint64(32), p & U32


def _rk(k, w, r):
    return np.uint64((k + r * w) & 0xFFFFFFFF)


def _env_head(env, blk, k0, k1):
    hi0, lo0 = _mul(M0, env)
    x = hi0 ^ np.asarray(blk, dtype=np.uint64) ^ _rk(k1, W1, 0)
    hi1, lo1 = _mul(M1, x)
    return hi1 ^ _rk(k0, W0, 1), lo1, lo0 ^ _rk(k1, W1, 1)


def _call_head(t, dp, k0):
    hi1, lo1 = _mul(M1, dp)
    c0 = hi1 ^ np.asarray(t, dtype=np.uint64) ^ _rk(k0, W0, 0)
    hi0, lo0 = _mul(M0, c0)
    return lo1, hi0, lo0


def _rk_heads(eh, uh, k0, k1):
    c0, c1, c2, c3 = eh[0] ^ uh[0], eh[1], eh[2] ^ uh[1], uh[2]
    for r in range(2, 10):
        hi0, lo0 = _mul(M0, c0)
        hi1, lo1 = _mul(M1, c2)
        c0, c1, c2, c3 = hi1 ^ c1 ^ _rk(k0, W0, r), lo1, hi0 ^ c3 ^ _rk(k1, W1, r), lo0
    return tuple(x.astype(np.uint32) for x in (c0, c1, c2, c3))


def test_philox_heads_equal_full_philox():
    rng = np.random.default_rng(7)
    for _ in range(20):
        k0, k1 = (int(x) for x in rng.integers(0, 1 << 32, 2))
        n = 4096
        env, t, blk = (rng.integers(0, 1 << 32, n, dtype=np.uint64) for _ in range(3))
        dp = rng.integers(0, 8, n, dtype=np.uint64) | (rng.integers(0, 3, n, dtype=np.uint64) << np.uint64(16))
        blk[: n // 2] = np.arange(n // 2, dtype=np.uint64) % 4            # the C = 16 callers' blocks 0 and 1, and more
        ref = px.philox4x32_10(env, t, dp, blk, k0, k1)
        got = _rk_heads(_env_head(env, blk, k0, k1), _call_head(t, dp, k0), k0, k1)
        for r, g in zip(ref, got):
            assert np.array_equal(r, g)


def test_lane_threshold_compare():
    """lanes_below: lane 2j + 1 (high half of word j) is below thr iff word < thr << 16; lane 2j iff word << 16 < thr
    << 16; thr = 65536 sets the lane unconditionally and thr = 0 never does."""
    rng = np.random.default_rng(3)
    w = rng.integers(0, 1 << 32, 100000, dtype=np.uint64)
    for thr in (0, 1, 2, 255, 32768, 65535, 65536, int(rng.integers(0, 65537))):
        lt = 0 if thr >= 65536 else thr << 16
        every = thr >= 65536
        hi = (w < lt) | every
        lo = (((w << np.uint64(16)) & U32) < lt) | every
        assert np.array_equal(hi, (w >> np.uint64(16)) < thr)
        assert np.array_equal(lo, (w & np.uint64(0xFFFF)) < thr)
