"""The returns stage of the PPO learners against a float64 restatement of the reference in the kernels' layout.

``returns_scan_kernel`` (raw / stats / emit, atomics or deterministic per-warp partials), ``sum_partials_kernel``,
``norm_stats_kernel`` and ``normalize_kernel`` turn the rollout's integer rewards and critic values into the normalised
lambda-returns (compute_gae, d2d_ppo.py:100-110) and discounted returns (discount_rewards, :112-124).  The tests below
drive every public entry point at every row-batching remainder, column count and block / grid-stride size, with the
learners' flag combinations, emulated multi-rank shard splits, the all-columns normalise gate and deterministic mode.

Tolerances (each derived from the error source it allows, nothing else):
* raw float64 outputs: RAW_TOL of the column's magnitude.  The kernel contracts ``r + gamma v' - v``, ``delta + gl gae``
  and ``r + run gamma`` into FMAs where numpy rounds every product, so it is not bit-exact.  Each row adds a few float64
  ulps of the column's magnitude and the scans damp older errors by gamma lambda or gamma per row, so the error stays
  below ~2 / (1 - gamma) ulps (200 ulps = 2e-14 at gamma = 0.99).  1e-12 leaves room for that and is still 1e-7 of
  any error a wrong row, column or quirk would make.
* statistics: each (sum, sum of squares) entry within RAW_TOL x rows x (magnitude or magnitude^2): the raw error above
  per row, plus summation-order rounding far below it, plus one fp32 ulp for each return whose raw value sits that
  close to an fp32 rounding boundary (``_bounds``).  Means and variances follow from those (``_stat_bounds``).
* normalised fp32 outputs: the float64 reference normalised once and rounded once, against which the kernel may differ
  by the fp32 roundings its documented arithmetic makes and by its statistics' errors (``_emit_bound``), and the
  project's 1e-5 norm-wise ``rel_err``.  Separately, the kernel's fp32 outputs are restated exactly from its own raw
  outputs and statistics: bit for bit for the float64 reciprocal multiply, within one ulp for the fp32 Markstein
  quotient.
"""
import numpy as np
import pytest
import torch

from _helpers import load_ppo_case, rel_err
from oracle import ppo_torch as P

TOL = 1e-5          # the project's norm-wise fp32 bound
RAW_TOL = 1e-12     # float64 scans, relative to the column's magnitude (see the module docstring)
GAMMA, LAM = 0.9, 0.97


# ---------------------------------------------------------------------------------------------
# float64 reference in the kernels' layout
# ---------------------------------------------------------------------------------------------
def returns_reference(reward, value, gamma, lam, last_shard=True):
    """compute_gae / discount_rewards (oracle/ppo_torch.py ``lambda_returns`` / ``discounted_returns``) in float64.

    reward: integer [T, B], shared by the columns as the kernels take it, or [T, n_cols, B]; value: [T, n_cols, B] or
    None (returns only, one column).  Env b's episode is t = 0 .. T - 1 of column b.  The reference's rows are
    episode-major, so its final row, the only one that keeps ``r - v`` (d2d_ppo.py:102), is env B - 1 at t = T - 1,
    and only if this block of envs holds the globally last env (``last_shard``).  Every other episode end gets
    ``(r - v) + v`` (done zeroes the bootstrap and the trace, not the delta).

    Returns a dict: ``adv`` / ``ret`` raw float64 [T, n_cols, B]; ``rows``; ``adv_mean`` / ``adv_std`` (numpy's
    population std of the float64 lambda-returns); ``ret_f32`` (the returns cast to fp32) and ``ret_mean`` /
    ``ret_std`` (its unbiased std, in float64); ``adv_norm`` / ``ret_norm`` (the reference's decision: EVERY column
    has a positive std); ``adv32`` / ``ret32``, the normalised values rounded once to fp32."""
    r = np.asarray(reward, dtype=np.float64)
    if r.ndim == 2:
        r = r[:, None, :]
    n_cols = r.shape[1] if value is None else value.shape[1]
    T, B = r.shape[0], r.shape[2]
    r = np.broadcast_to(r, (T, n_cols, B))
    v = np.zeros((T, n_cols, B)) if value is None else np.asarray(value, dtype=np.float64)
    adv, ret = np.empty((T, n_cols, B)), np.empty((T, n_cols, B))
    gae = r[-1] - v[-1]
    adv[-1] = gae + v[-1]
    if last_shard:
        adv[-1, :, -1] = r[-1, :, -1] - v[-1, :, -1]
        gae[:, -1] = 0.0
    run = r[-1].copy()
    ret[-1] = run
    for t in range(T - 2, -1, -1):
        gae = (r[t] + gamma * v[t + 1] - v[t]) + gamma * lam * gae
        adv[t] = gae + v[t]
        run = r[t] + run * gamma
        ret[t] = run

    def rows(x):   # [T, n_cols, B] -> the reference's episode-major [B * T, n_cols] (same summation order)
        return x.transpose(2, 0, 1).reshape(B * T, n_cols)
    a_rows = rows(adv)
    ret_f32 = ret.astype(np.float32)
    r_rows = rows(ret_f32).astype(np.float64)
    out = dict(adv=adv, ret=ret, ret_f32=ret_f32, rows=T * B, adv_mean=a_rows.mean(0), adv_std=a_rows.std(0),
               ret_mean=r_rows.mean(0), ret_std=r_rows.std(0, ddof=1))
    out["adv_norm"] = bool((out["adv_std"] > 0).all())
    out["ret_norm"] = bool((out["ret_std"] > 0).all())
    col = (None, slice(None), None)
    out["adv32"] = ((adv - out["adv_mean"][col]) / out["adv_std"][col] if out["adv_norm"] else adv).astype(np.float32)
    out["ret32"] = ((ret_f32 - out["ret_mean"][col]) / out["ret_std"][col] if out["ret_norm"] else
                    ret_f32).astype(np.float32)
    return out


def _env_minor(x, E, T):
    """[R = E * T, N] episode-major rows -> [T, N, E]."""
    return np.ascontiguousarray(x.reshape(E, T, x.shape[1]).transpose(1, 2, 0))


def _rows(x):
    """[T, N, E] -> [R = E * T, N] episode-major rows."""
    T, N, E = x.shape
    return x.transpose(2, 0, 1).reshape(E * T, N)


def _ulp32(x):
    return np.spacing(np.abs(np.asarray(x, dtype=np.float64)).astype(np.float32)).astype(np.float64)


def _assert_within(what, mine, ref, bound):
    mine, ref = np.asarray(mine, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    assert mine.shape == ref.shape, (what, mine.shape, ref.shape)
    err = np.abs(mine - ref)
    bad = ~(err <= bound)
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, err / np.maximum(bound, 1e-300), 0)), err.shape)
        raise AssertionError(f"{what}: {int(bad.sum())} of {err.size} entries out of bounds; worst at {i}: "
                             f"{mine[i]!r} vs {ref[i]!r} (bound {np.broadcast_to(bound, err.shape)[i]:.3e})")


def _ret32_bound(ref):
    """Elementwise bound of the kernel's fp32 normalised returns against ``ref['ret32']``: (x - m) / s in fp32 with
    m and s rounded to fp32 first (torch's tensors) is three roundings of the result (subtraction, s, quotient:
    3 ulps), plus half an ulp of m over s; the kernel's own cast of its raw return may land one fp32 ulp away where
    the raw differs by RAW_TOL from a rounding boundary (one ulp of x over s)."""
    if not ref["ret_norm"]:
        return _ulp32(ref["ret_f32"])
    m, s = ref["ret_mean"][None, :, None], ref["ret_std"][None, :, None]
    return 3 * _ulp32(ref["ret32"]) + (_ulp32(ref["ret_f32"]) + _ulp32(m)) / s


# ---------------------------------------------------------------------------------------------
# CPU: the reference is the reference's semantics
# ---------------------------------------------------------------------------------------------
def test_reference_matches_golden_and_oracle():
    """Against the reference's own outputs (tests/golden/ppo_returns.npz, written by the unmodified compute_gae /
    discount_rewards) and against the torch oracle on random shared-reward data."""
    g = load_ppo_case("returns")
    for tag in ("a", "b", "c"):
        T = int(g[f"{tag}/T"])
        E = g[f"{tag}/rewards"].shape[0] // T
        reward, value = _env_minor(g[f"{tag}/rewards"], E, T), _env_minor(g[f"{tag}/values"], E, T)
        for gamma in (0.6, 0.99):
            ref = returns_reference(reward, value, gamma, 0.97)
            assert ref["adv_norm"] and ref["ret_norm"]
            # same operations in the same order as numpy's compute_gae: bit for bit
            assert np.array_equal(_rows(ref["adv32"]), g[f"{tag}/g{gamma}/adv"]), (tag, gamma)
            # torch normalises in fp32 with fp32 mean / std: the kernels' fp32 bound
            ref32 = _env_minor(g[f"{tag}/g{gamma}/ret"], E, T)
            _assert_within(f"{tag} g{gamma} ret", ref32, ref["ret32"], _ret32_bound(ref))
    # zero-std columns (gamma = 0, constant reward, zero values): no normalisation of either output
    ref = returns_reference(np.ones((4, 2, 3)), np.zeros((4, 2, 3)), 0.0, 0.97)
    assert not ref["adv_norm"] and not ref["ret_norm"]
    assert np.array_equal(_rows(ref["adv32"]), g["deg/adv"]) and np.array_equal(_rows(ref["ret32"]), g["deg/ret"])

    rng = np.random.default_rng(3)
    for T, n_cols, B in ((9, 3, 5), (1, 2, 7), (25, 1, 4)):
        reward = rng.integers(0, 9, (T, B)).astype(np.int32)
        value = rng.standard_normal((T, n_cols, B)).astype(np.float32)
        for gamma in (0.6, 0.99):
            ref = returns_reference(reward, value, gamma, 0.97)
            r_rows = _rows(np.broadcast_to(reward[:, None, :], (T, n_cols, B)))
            dones = [(i % T) == T - 1 for i in range(B * T)]
            adv = P.lambda_returns(r_rows, dones, _rows(value), gamma, 0.97).numpy()
            assert np.array_equal(_rows(ref["adv32"]), adv), (T, n_cols, B, gamma)
            ret = P.discounted_returns(r_rows, gamma, dones).numpy()
            _assert_within(f"random ret {T} {n_cols} {B}", _env_minor(ret, B, T), ref["ret32"],
                           _ret32_bound(ref))
    # not the last shard: the final row is an ordinary episode end
    ref = returns_reference(reward, value, 0.6, 0.97, last_shard=False)
    assert np.array_equal(ref["adv"][-1], (reward[-1][None] - value[-1].astype(np.float64)) + value[-1])


# ---------------------------------------------------------------------------------------------
# GPU: the kernels against the reference
# ---------------------------------------------------------------------------------------------
def _grid_cap_envs():
    """Envs one launch covers before returns_scan_kernel's grid-stride loop wraps (grid_for: SMs x 8 blocks x 128)."""
    return torch.cuda.get_device_properties(0).multi_processor_count * 8 * 128


def _inputs(T, n_cols, B, seed, r_max=8, mixed=False):
    rng = np.random.default_rng(seed)
    reward = rng.integers(0, r_max + 1, (T, B)).astype(np.int32)
    value = rng.standard_normal((T, n_cols, B))
    if mixed:   # critic values of both signs over 4.5 decades
        value *= 10.0 ** rng.uniform(-2.0, 2.5, value.shape)
    return reward, value.astype(np.float32)


def _dev(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def _np(t):
    return t.cpu().numpy()


def _bounds(ref, value):
    """What the float64 errors are relative to, per column.
    scale: the largest |output| or |value| of the column.
    slack: for the returns, the sum of one fp32 ulp over the entries whose raw value lies within RAW_TOL x scale of an
    fp32 rounding boundary: there the kernel's own cast to fp32 (its statistics are of the cast returns) may round
    the other way.  0 for the lambda-returns, which are summed in float64."""
    s = np.maximum(np.abs(ref["adv"]).max(axis=(0, 2)), np.abs(ref["ret"]).max(axis=(0, 2)))
    if value is not None:
        s = np.maximum(s, np.abs(value).max(axis=(0, 2)))
    scale = np.maximum(s, 1.0)
    x, a = np.abs(ref["ret"]), np.abs(ref["ret_f32"])
    up = np.spacing(a).astype(np.float64)
    down = (a - np.nextafter(a, np.float32(0))).astype(np.float64)
    half = np.where(x > a, up, down) / 2                       # distance from the fp32 value to the boundary x faces
    near = half - np.abs(x - a) <= RAW_TOL * scale[None, :, None]
    return {"scale": scale, "adv": np.zeros_like(scale), "ret": (near * up).sum(axis=(0, 2))}


def _stat_bounds(ref, bd, key):
    """(mean, variance) error bounds of norm_stats_kernel's outputs: the sums' bounds (``_check_stats``) over the
    row count; the variance (sum^2 - n mean^2) / d also carries n x 2 mean x the mean's error.  The one-pass
    difference rounds at ~1e-16 of n x the mean square, far inside these."""
    n, scale, slack = ref["rows"], bd["scale"], bd[key]
    d = n if key == "adv" else n - 1
    return RAW_TOL * scale + slack / n, (4 * RAW_TOL * n * scale * scale + 4 * scale * slack) / d


def _check_stats(what, stats, ref, bd, want_adv, want_ret):
    """[n_cols, 4] sums (adv, adv^2, fp32 ret, fp32 ret^2) against the reference's: each row's raw error (RAW_TOL x
    scale) times the rows, plus the cast slack of the returns; a quantity not asked for is exactly 0."""
    n, scale = ref["rows"], bd["scale"]
    for k, (on, key, x) in enumerate(((want_adv, "adv", ref["adv"]), (want_ret, "ret", ref["ret_f32"].astype(np.float64)))):
        s, q = stats[:, 2 * k], stats[:, 2 * k + 1]
        if not on:
            assert not s.any() and not q.any(), (what, key, s, q)
            continue
        _assert_within(f"{what} {key} sum", s, x.sum(axis=(0, 2)), RAW_TOL * n * scale + bd[key])
        _assert_within(f"{what} {key} sumsq", q, (x * x).sum(axis=(0, 2)),
                       2 * RAW_TOL * n * scale * scale + 2 * scale * bd[key])


def _check_norm(what, norm, ref, bd, key):
    """(mean, std, flags) of norm_stats_kernel against the reference: mean and variance within ``_stat_bounds``
    (|std - std_ref| (std + std_ref) = |var - var_ref|), the flags exactly."""
    mean, std, flags = (_np(t) for t in norm)
    mean_err, var_err = _stat_bounds(ref, bd, key)
    _assert_within(f"{what} {key} mean", mean, ref[f"{key}_mean"], mean_err)
    sr = ref[f"{key}_std"]
    _assert_within(f"{what} {key} std", std, sr, var_err / np.maximum(std + sr, 1e-300))
    assert (flags == int(ref[f"{key}_norm"])).all(), (what, key, flags, ref[f"{key}_norm"])


def _emit_bound(ref, bd, key):
    """Elementwise bound of a normalised fp32 output y = (x - m) / s against the reference's ``{key}32``.
    adv: one ulp for the cast (the kernel's float64 value may sit on the other side of a rounding boundary) plus
    (raw error + mean error) / s + |y| x the std's relative error (var_err / s^2 bounds it twice over).
    ret: ``_ret32_bound`` (the fp32 arithmetic) plus the mean and std errors the same way."""
    ref32 = ref[f"{key}32"]
    if not ref[f"{key}_norm"]:
        return _ulp32(ref32) + (RAW_TOL * bd["scale"][None, :, None] if key == "adv" else 0.0)
    mean_err, var_err = (e[None, :, None] for e in _stat_bounds(ref, bd, key))
    s = ref[f"{key}_std"][None, :, None]
    stat = mean_err / s + np.abs(ref32) * var_err / (s * s)
    if key == "adv":
        return _ulp32(ref32) + RAW_TOL * bd["scale"][None, :, None] / s + stat
    return _ret32_bound(ref) + stat


def _check_emit(what, out, raw, norm, ref, bd, key):
    """The normalised fp32 output of one quantity.
    1. Restated from the kernel's own raw output and statistics.  adv: (raw - mean) * (1 / std) in float64, cast:
       bit for bit.  ret: (fl32(raw) - fl32(mean)) / fl32(std) in fp32; the kernel's Markstein quotient is correctly
       rounded except for divisors with an all-ones mantissa, where it may be one ulp off.
    2. Against the reference within ``_emit_bound``, and the project's norm-wise bound."""
    out, raw = _np(out), _np(raw)
    mean, std, flags = (_np(t)[None, :, None] for t in norm)
    on = bool(flags.all())
    assert flags.all() == flags.any()
    if key == "adv":
        assert np.array_equal(out, ((raw - mean) * (1.0 / std) if on else raw).astype(np.float32)), what
    else:
        xf = raw.astype(np.float32)
        if on:
            q = (xf - mean.astype(np.float32)) / std.astype(np.float32)
            _assert_within(f"{what} ret restated", out, q, _ulp32(q))
        else:
            assert np.array_equal(out, xf), what
    _assert_within(f"{what} {key} normalised", out, ref[f"{key}32"], _emit_bound(ref, bd, key))
    assert rel_err(out, ref[f"{key}32"]) < TOL, what


def _check_stage(dev, reward, value, gamma, lam, want_adv=True, want_ret=True, last_shard=True, what=""):
    """Every entry point on one block of envs against the reference, for one flag combination:
    returns_scan (raw + one-pass statistics) -> normalize, and returns_stats -> returns_norm_stats -> returns_emit.
    Returns (reference, kernel statistics, (adv norm, ret norm), (adv out, ret out))."""
    from d2d_ppo_b200.algorithms._nets import normalize, returns_emit, returns_norm_stats, returns_scan, returns_stats
    T, B = reward.shape
    val = value if want_adv else None
    ref = returns_reference(reward, val, gamma, lam, last_shard)
    bd = _bounds(ref, val)
    r_d, v_d = _dev(reward, dev), (None if val is None else _dev(val, dev))

    adv_raw, ret_raw, stats1 = returns_scan(r_d, v_d, gamma, lam, last_shard, want_adv, want_ret)
    assert (adv_raw is not None) == want_adv and (ret_raw is not None) == want_ret
    for on, raw, key in ((want_adv, adv_raw, "adv"), (want_ret, ret_raw, "ret")):
        if on:
            _assert_within(f"{what} {key} raw", _np(raw), ref[key], RAW_TOL * bd["scale"][None, :, None])
    _check_stats(f"{what} one-pass", _np(stats1), ref, bd, want_adv, want_ret)
    stats = returns_stats(r_d, v_d, gamma, lam, last_shard, want_adv, want_ret)
    _check_stats(f"{what} two-pass", _np(stats), ref, bd, want_adv, want_ret)

    norm_a, norm_r = returns_norm_stats(stats, ref["rows"])
    adv_out, ret_out = returns_emit(r_d, v_d, gamma, lam, last_shard, norm_a if want_adv else None,
                                    norm_r if want_ret else None)
    for on, norm, out, raw, key, fp32 in ((want_adv, norm_a, adv_out, adv_raw, "adv", 0),
                                          (want_ret, norm_r, ret_out, ret_raw, "ret", 1)):
        if not on:
            assert out is None
            continue
        _check_norm(what, norm, ref, bd, key)
        _check_emit(what, out, raw, norm, ref, bd, key)
        # the one-pass path (float64 outputs, then normalize_kernel) gives the same bits as the two-pass one
        assert torch.equal(normalize(raw, *norm, fp32), out), (what, key)
    return ref, stats, (norm_a, norm_r), (adv_out, ret_out)


# the learners' flag combinations: iPPO asks for both with N columns (ippo.py:46-51); D2DPPO for the returns alone
# without values (d2d_ppo.py:45-49) and for the lambda-returns alone (:68-71)
COMBOS = {"both": (True, True), "adv_only": (True, False), "ret_only": (False, True)}

# T: every (T - 1) % 6 and 0, 1, 2 and 3+ whole 6-row batches of the two register buffers (T = 1: episode end only)
T_SWEEP = [(T, 3, 129) for T in (1, 2, 6, 7, 8, 12, 13, 14, 19, 25, 200)]
# columns x blocks: one warp, several warps, several blocks, 64 columns (D2D_MAX_AGENTS, and the 64 threads of
# norm_stats_kernel), and "cap": 77 envs more than one launch covers, so the grid-stride loop runs a second time
COL_SWEEP = [(13, 1, 1), (13, 1, 31), (13, 6, 31), (13, 64, 31), (8, 64, 129), (13, 3, 4096), (8, 64, 4096),
             (7, 1, 65536), (13, 6, 65536), (7, 1, "cap"), (3, 2, "cap")]


@pytest.mark.gpu
@pytest.mark.parametrize("T,n_cols,B", T_SWEEP + COL_SWEEP)
def test_returns_stage_matches_reference(T, n_cols, B, cuda_device):
    if B == "cap":
        B = _grid_cap_envs() + 77
    reward, value = _inputs(T, n_cols, B, seed=T * 1000 + n_cols)
    for name, (want_adv, want_ret) in COMBOS.items():
        _check_stage(cuda_device, reward, value, GAMMA, LAM, want_adv, want_ret, what=f"T={T} N={n_cols} B={B} {name}")


@pytest.mark.gpu
@pytest.mark.parametrize("B", [129, 4096])
def test_long_episodes_large_returns(B, cuda_device):
    """gamma = 0.99 over 200 rows with rewards up to 64: early rows sum the whole discounted future (returns in the
    thousands), and values of both signs over 4.5 decades; this is where the one-pass (sum, sum of squares)
    statistics lose the most digits."""
    reward, value = _inputs(200, 3, B, seed=B, r_max=64, mixed=True)
    for name, (want_adv, want_ret) in COMBOS.items():
        ref, *_ = _check_stage(cuda_device, reward, value, 0.99, 0.97, want_adv, want_ret, what=f"B={B} {name}")
    assert np.abs(ref["ret"]).max() > 1000


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 3, 8])
def test_sharded_run_matches_single_call(K, cuda_device):
    """A K-rank run on one GPU: contiguous uneven shards (_dist.shard), per-shard statistics with only the last shard
    keeping the final-row quirk, the summed statistics over the global row count, then per-shard emits."""
    from d2d_ppo_b200.algorithms import _dist
    from d2d_ppo_b200.algorithms._nets import returns_emit, returns_norm_stats, returns_scan, returns_stats
    dev = cuda_device
    T, n_cols, B = 13, 3, 1001
    assert B % K
    reward, value = _inputs(T, n_cols, B, seed=K)
    ref, _, single_norm, single_out = _check_stage(dev, reward, value, GAMMA, LAM, what=f"K={K} single")
    bd = _bounds(ref, value)
    shards = [_dist.shard(B, k, K) for k in range(K)]
    assert len({c for _, c in shards}) == 2      # uneven

    def part(k):
        off, cnt = shards[k]
        return _dev(reward[:, off:off + cnt], dev), _dev(value[:, :, off:off + cnt], dev)

    def run(last):   # last(k): the last_shard flag of shard k
        stats = sum(returns_stats(*part(k), GAMMA, LAM, last(k)) for k in range(K))
        norm = returns_norm_stats(stats, T * B)
        outs = [returns_emit(*part(k), GAMMA, LAM, last(k), *norm) for k in range(K)]
        return stats, norm, [torch.cat([o[i] for o in outs], dim=2) for i in range(2)]

    stats, norm, (adv, ret) = run(lambda k: k == K - 1)
    _check_stats(f"K={K}", _np(stats), ref, bd, True, True)
    for key, norm_k, out in (("adv", norm[0], adv), ("ret", norm[1], ret)):
        _check_norm(f"K={K}", norm_k, ref, bd, key)
        _assert_within(f"K={K} {key}", _np(out), ref[f"{key}32"], _emit_bound(ref, bd, key))
        assert rel_err(_np(out), ref[f"{key}32"]) < TOL
    # with the single call's statistics, every env's outputs are the single call's, bit for bit
    outs = [returns_emit(*part(k), GAMMA, LAM, k == K - 1, *single_norm) for k in range(K)]
    for i in range(2):
        assert torch.equal(torch.cat([o[i] for o in outs], dim=2), single_out[i]), (K, i)

    # negative check: with last_shard = 0 everywhere the quirk is gone, and the final row is an ordinary episode end
    ref0 = returns_reference(reward, value, GAMMA, LAM, last_shard=False)
    assert (np.abs(ref0["adv"][-1, :, -1] - ref["adv"][-1, :, -1]) > 1e-3).all()
    raw = torch.cat([returns_scan(*part(k), GAMMA, LAM, 0)[0] for k in range(K)], dim=2)
    _assert_within(f"K={K} no quirk", _np(raw), ref0["adv"], RAW_TOL * bd["scale"][None, :, None])
    _, norm0, (adv0, _) = run(lambda k: False)
    _check_norm(f"K={K} no quirk", norm0[0], ref0, _bounds(ref0, value), "adv")
    _assert_within(f"K={K} no quirk adv", _np(adv0), ref0["adv32"], _emit_bound(ref0, _bounds(ref0, value), "adv"))


@pytest.mark.gpu
def test_one_constant_column_switches_normalisation_off(cuda_device):
    """The reference normalises only if EVERY column has a positive std, for the lambda-returns and the returns
    independently.  lam = 0 and a constant reward make a lambda-return column with zero values exactly constant
    (r + gamma * 0 at every row, r - 0 at the quirk row), while columns with values vary with gamma v(t + 1); the
    returns do not depend on the values and vary with t, so they still normalise."""
    T, n_cols, B = 9, 4, 33
    reward, value = _inputs(T, n_cols, B, seed=7)
    reward[:] = 3
    value[:, 2] = 0.0
    ref, _, (norm_a, norm_r), _ = _check_stage(cuda_device, reward, value, GAMMA, 0.0, what="constant column")
    assert ref["adv_std"][2] == 0.0 and (np.delete(ref["adv_std"], 2) > 0.1).all()
    assert not _np(norm_a[2]).any() and _np(norm_r[2]).all()
    # the same columns without the constant one normalise
    _, _, (norm_a, _), _ = _check_stage(cuda_device, reward, np.delete(value, 2, axis=1), GAMMA, 0.0,
                                        what="variable columns")
    assert _np(norm_a[2]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("constant", ["adv", "ret"])
def test_norm_stats_gate_is_per_quantity(constant, cuda_device):
    """norm_stats_kernel on summed statistics as they arrive from the ranks: one exactly constant column of one
    quantity switches off that quantity's normalisation for every column, and only that quantity's.  (The kernels'
    returns are the same in every column, so a single constant return column can only come from constructed sums.)"""
    from d2d_ppo_b200.algorithms._nets import returns_norm_stats
    rng = np.random.default_rng(11)
    n_cols, rows = 5, 300
    x = {k: rng.standard_normal((rows, n_cols)).astype(np.float32).astype(np.float64) * 4 + 2 for k in ("adv", "ret")}
    x[constant][:, 3] = 2.5
    stats = np.stack([x["adv"].sum(0), (x["adv"] ** 2).sum(0), x["ret"].sum(0), (x["ret"] ** 2).sum(0)], axis=1)
    norm = dict(zip(("adv", "ret"), returns_norm_stats(_dev(stats, cuda_device), rows)))
    for key, ddof in (("adv", 0), ("ret", 1)):
        mean, std, flags = (_np(t) for t in norm[key])
        # float64 rounding of 300 terms of magnitude < 20: the mean within 1e-14, the variance within 1e-11
        _assert_within(f"{key} mean", mean, x[key].mean(0), 1e-14)
        sr = x[key].std(0, ddof=ddof)
        assert (sr[3] == 0.0) == (key == constant)
        _assert_within(f"{key} std", std, sr, 1e-11 / np.maximum(std + sr, 1e-300))
        assert (flags == int(key != constant)).all(), (key, flags)


@pytest.mark.gpu
def test_gate_threshold_is_relative_to_the_mean_square(cuda_device):
    """The one-pass (sum, sum of squares) variance of an exactly constant column is rounding noise of order
    1e-16 x rows x mean^2 where numpy gives exactly 0, so norm_stats_kernel normalises only if var > 1e-9 x the mean
    square.  That departs from numpy (std > 0) for columns whose std is below sqrt(1e-9) ~ 3.2e-5 of their RMS:
    such a column is left unnormalised although numpy would divide by its tiny std.  This is intended: it is the
    price of never normalising a constant column by noise.  With T >= 2 and the learners' discounts (0.2 to 0.99) even
    a constant reward gives returns that differ by a factor 1 + gamma within each episode, far above the threshold.
    Pinned here with integer rewards c +- 1 and gamma = 0, where every return and every sum is exact:
    std / RMS = 1e-5 stays unnormalised, 1e-4 normalises."""
    from d2d_ppo_b200.algorithms._nets import returns_norm_stats, returns_stats
    dev = cuda_device
    T, B = 4, 64
    value = np.zeros((T, 1, B), dtype=np.float32)
    sign = np.where((np.arange(T)[:, None] + np.arange(B)[None, :]) % 2 == 1, 1, -1)
    for c, below in ((100000, True), (10000, False)):
        reward = (c + sign).astype(np.int32)
        ref = returns_reference(reward, value, 0.0, LAM)
        assert np.array_equal(ref["adv"][:, 0], reward) and np.array_equal(ref["ret"][:, 0], reward)
        assert ref["adv_norm"] and ref["ret_norm"]           # numpy / torch: std > 0, normalise
        assert (ref["adv_std"][0] / c < 3.16e-5) == below
        stats = returns_stats(_dev(reward, dev), _dev(value, dev), 0.0, LAM, 1)
        (am, asd, af), (rm, rsd, rf) = returns_norm_stats(stats, T * B)
        assert am.item() == c and asd.item() == 1.0 and rm.item() == c and rsd.item() == np.sqrt(T * B / (T * B - 1))
        assert af.item() == rf.item() == int(not below), (c, af.item(), rf.item())
        if not below:
            _check_stage(dev, reward, value, 0.0, LAM, what=f"c={c}")


@pytest.fixture
def deterministic():
    import d2d_ppo_b200
    before = d2d_ppo_b200.are_deterministic_algorithms_enabled()
    d2d_ppo_b200.use_deterministic_algorithms(True)
    try:
        yield d2d_ppo_b200.use_deterministic_algorithms
    finally:
        d2d_ppo_b200.use_deterministic_algorithms(before)


@pytest.mark.gpu
@pytest.mark.parametrize("T,n_cols,B,mixed", [(13, 6, 31, False), (8, 64, 4096, False), (200, 3, 129, True),
                                              (7, 2, "cap", False)])
def test_deterministic_mode(T, n_cols, B, mixed, deterministic, cuda_device):
    """kScanPartials: per-warp sums reduced by sum_partials_kernel in a fixed order.  The statistics are bit-identical
    across calls and between the one-pass and two-pass scans, agree with the default mode's atomics within the
    statistics bound, and the whole stage matches the reference as in the default mode."""
    from d2d_ppo_b200.algorithms._nets import returns_scan, returns_stats
    if B == "cap":
        B = _grid_cap_envs() + 77
    n_warps = min(-(-B // 128), torch.cuda.get_device_properties(0).multi_processor_count * 8) * 4
    reward, value = _inputs(T, n_cols, B, seed=T + B, r_max=64 if mixed else 8, mixed=mixed)
    gamma = 0.99 if mixed else GAMMA
    ref, stats, *_ = _check_stage(cuda_device, reward, value, gamma, LAM, what="deterministic")
    r_d, v_d = _dev(reward, cuda_device), _dev(value, cuda_device)
    for _ in range(2):
        assert torch.equal(returns_stats(r_d, v_d, gamma, LAM, 1), stats)
        assert torch.equal(returns_scan(r_d, v_d, gamma, LAM, 1)[2], stats)
    deterministic(False)
    atomics = returns_stats(r_d, v_d, gamma, LAM, 1)
    _check_stats("atomics", _np(atomics), ref, _bounds(ref, value), True, True)
    # both add the same per-warp sums, in different orders: a sum of n_warps terms moves by at most
    # n_warps ulps of the sum of their magnitudes under reordering, each way
    x = (np.abs(ref["adv"]), ref["adv"] ** 2, np.abs(ref["ret_f32"].astype(np.float64)), ref["ret_f32"].astype(np.float64) ** 2)
    mag = np.stack([m.sum(axis=(0, 2)) for m in x], axis=1)
    _assert_within("deterministic vs atomics", _np(stats), _np(atomics), 2 * n_warps * 2.0 ** -52 * mag)


@pytest.mark.gpu
def test_bad_arguments_raise_before_any_launch(cuda_device):
    from d2d_ppo_b200 import _lib as L
    from d2d_ppo_b200.algorithms._nets import returns_emit, returns_norm_stats, returns_scan, returns_stats
    dev = cuda_device
    T, B = 5, 8
    r = torch.zeros((T, B), dtype=torch.int32, device=dev)
    v = torch.zeros((T, 2, B), dtype=torch.float32, device=dev)
    v65 = torch.zeros((T, 65, B), dtype=torch.float32, device=dev)
    stats = torch.ones((2, 4), dtype=torch.float64, device=dev)
    na, nr = returns_norm_stats(stats, 10)
    torch.cuda.synchronize()
    calls = {
        "scan T=0": lambda: returns_scan(r[:0], v[:0], GAMMA, LAM, 1),
        "scan B=0": lambda: returns_scan(r[:, :0], v[:, :, :0], GAMMA, LAM, 1),
        "scan n_cols=65": lambda: returns_scan(r, v65, GAMMA, LAM, 1),
        "scan adv without values": lambda: returns_scan(r, None, GAMMA, LAM, 1),
        "stats T=0": lambda: returns_stats(r[:0], v[:0], GAMMA, LAM, 1),
        "stats B=0": lambda: returns_stats(r[:, :0], v[:, :, :0], GAMMA, LAM, 1),
        "stats n_cols=65": lambda: returns_stats(r, v65, GAMMA, LAM, 1),
        "stats adv without values": lambda: returns_stats(r, None, GAMMA, LAM, 1),
        "norm_stats rows=1": lambda: returns_norm_stats(stats, 1),
        "norm_stats n_cols=65": lambda: returns_norm_stats(torch.ones((65, 4), dtype=torch.float64, device=dev), 10),
        "emit T=0": lambda: returns_emit(r[:0], v[:0], GAMMA, LAM, 1, na, nr),
        "emit B=0": lambda: returns_emit(r[:, :0], v[:, :, :0], GAMMA, LAM, 1, na, nr),
        "emit n_cols=65": lambda: returns_emit(r, v65, GAMMA, LAM, 1, na, nr),
        "emit adv without values": lambda: returns_emit(r, None, GAMMA, LAM, 1, na, None),
    }
    for what, call in calls.items():
        n0 = L.launch_count()
        with pytest.raises(L.D2DError) as e:
            call()
        assert e.value.code == L.ERR_INVALID, what
        assert L.launch_count() == n0, what
