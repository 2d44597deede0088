"""CombinatorialEnv, N <= 8, C = 4 or 8: d2d_env_run_random_access runs the steps of an episode inside ONE kernel with
the env state in registers (comb_run_kernel).  Bit-identical to the same call with the multi-step kernel switched off
(one comb_step_kernel launch per step), and to the numpy oracle."""
import numpy as np
import pytest

from _helpers import to_np

pytestmark = pytest.mark.gpu


def _kwargs(N, C, D, traffic, T):
    """N devices, C channels, deadlines D and D - 5 alternating (D = 7: 8-byte records, D = 14: 16-byte records)."""
    rng = np.random.default_rng(N * 100 + C + D)
    kw = dict(n_agents=N, n_channels=C, deadlines=np.array([D if k % 2 == 0 else D - 5 for k in range(N)]),
              lbdas=np.array([0.3] * N), episode_length=T, traffic_model=traffic,
              channel_switch=rng.uniform(0.0, 0.4, (N, C)), homogeneous_size=(D == 14))
    if traffic == "periodic":
        kw.update(period=3, arrival_probs=np.array([0.7] * N), offsets=np.arange(N) % 3)
    if traffic == "heterogeneous":
        kw.update(period=np.array([4] * N), arrival_probs=np.array([0.6] * N), offsets=np.arange(N) % 4,
                  periodic_devices=[k for k in (1, 3, 6) if k < N])
    return kw


def _launches(t0, n, T):
    """(resets, episode segments) of run_random_access(n, auto_reset=True) started at timestep t0."""
    t, resets, segments, prev = t0, 0, 0, None
    for _ in range(n):
        if t >= T:
            t, resets = 0, resets + 1
        if prev is None or t == 0:
            segments += 1
        prev = t
        t += 1
    return resets, segments


def _run(kw, B, multi, device, out_state=False):
    """One fixed sequence of run_random_access calls with the multi-step kernel switched on or off."""
    import torch
    from d2d_ppo_b200 import _lib as L
    from d2d_ppo_b200.envs import CombinatorialEnv
    T, tp = kw["episode_length"], 0.3
    L.set_kernel_switch(L.SWITCH_ENV_MULTISTEP, multi)
    try:
        e = CombinatorialEnv(n_envs=B, device=device, seed=17, env_offset=1000, **kw)
        R = e.obs_layout[0]
        e.reset()
        first = torch.zeros(B, dtype=torch.int32, device=device)
        assert e.run_random_access(tp, 3, out_reward=first) == 3                        # start mid-episode
        n = 2 * T + 5                                                                  # crosses two resets
        obs = torch.full((n, R, B), -5.0, device=device)
        rew = torch.full((n, B), -7, dtype=torch.int32, device=device)
        state = torch.zeros((n, e.state_space.shape[0], B), device=device) if out_state else None
        before = L.launch_count()
        assert e.run_random_access(tp, n, auto_reset=True, out_obs=obs, obs_stride=R * B, out_reward=rew,
                                   reward_stride=B, out_state=state,
                                   state_stride=0 if state is None else state[0].numel()) == n
        launches = L.launch_count() - before
        done1 = to_np(e.done_tensor)
        # the same block every step: the final block holds the last step's rows; the reward is overwritten
        obs0 = torch.full((R, B), -5.0, device=device)
        rew0 = torch.full((B,), -7, dtype=torch.int32, device=device)
        assert e.run_random_access(tp, T - 2, auto_reset=True, out_obs=obs0, out_reward=rew0) == T - 2
        done2 = to_np(e.done_tensor)
        acc = torch.full((B,), 4, dtype=torch.int32, device=device)
        e.reset()
        assert e.run_random_access(tp, T + 3, out_reward=acc, accumulate=True) == T
        done3 = to_np(e.done_tensor)
        torch.cuda.synchronize()
        return dict(first=to_np(first), obs=to_np(obs), rew=to_np(rew), done1=done1, obs0=to_np(obs0),
                    rew0=to_np(rew0), done2=done2, acc=to_np(acc), done3=done3,
                    state=[to_np(x) for x in e._export()], t=e.timestep, episode=e.episode, launches=launches)
    finally:
        L.set_kernel_switch(L.SWITCH_ENV_MULTISTEP, 1)


@pytest.mark.parametrize("B", [333, 40000])
@pytest.mark.parametrize("N,C,D,traffic", [(1, 4, 7, "aperiodic"), (4, 8, 14, "periodic"),
                                           (6, 8, 14, "heterogeneous"), (6, 4, 7, "periodic"),
                                           (8, 4, 14, "aperiodic"), (8, 8, 7, "heterogeneous")])
def test_comb_multistep_kernel_equals_step_kernels(N, C, D, traffic, B, cuda_device):
    """Per-step observations (stride R * B), the final block at stride 0, rewards in the per-step, overwrite and
    accumulate forms, done flags, records, channel masks and disc / recv counters: switch on == switch off."""
    T = 11
    kw = _kwargs(N, C, D, traffic, T)
    on, off = _run(kw, B, 1, cuda_device), _run(kw, B, 0, cuda_device)
    for key in ("first", "obs", "rew", "done1", "obs0", "rew0", "done2", "acc", "done3"):
        assert np.array_equal(on[key], off[key]), key
    for x, y in zip(on["state"], off["state"]):
        assert np.array_equal(x, y)
    assert on["t"] == off["t"] and on["episode"] == off["episode"]
    assert (on["obs"] != -5.0).all() and (on["obs0"] != -5.0).all() and (on["rew"] > 0).any()
    assert not on["done1"].any() and not on["done2"].any() and on["done3"].all()
    # resets + one launch per episode segment with the switch on, one launch per step with it off
    resets, segments = _launches(3, 2 * T + 5, T)
    assert on["launches"] == resets + segments and off["launches"] == resets + 2 * T + 5


@pytest.mark.parametrize("case", ["c16", "out_state"])
def test_comb_multistep_fallback_launches_per_step(case, cuda_device):
    """C = 16 and runs that emit state rows keep one comb_step_kernel launch per step."""
    T = 11
    kw = _kwargs(6, 16 if case == "c16" else 8, 14, "aperiodic", T)
    on = _run(kw, 333, 1, cuda_device, out_state=(case == "out_state"))
    resets, _ = _launches(3, 2 * T + 5, T)
    assert on["launches"] == resets + 2 * T + 5


def test_comb_multistep_matches_oracle(cuda_device):
    """The bench's config (setup_8_channels, N = 6, C = 8, homogeneous observation size) with the fused random-access
    policy, one episode in one launch: every step's observation rows and rewards, and the final state, equal the numpy
    oracle fed the action bits of the Philox policy stream."""
    import torch
    from d2d_ppo_b200 import _lib as L, presets
    from d2d_ppo_b200.envs import CombinatorialEnv
    from oracle import philox_np as px
    from oracle.envs_np import CombinatorialOracle, PhiloxSource
    B, T, seed, off, tp = 1000, 16, 23, 5, 0.25
    kw = presets.combinatorial_kwargs("setup_8_channels", load=0.5, episode_length=T)
    N, C = kw["n_agents"], kw["n_channels"]
    env = CombinatorialEnv(n_envs=B, device=cuda_device, seed=seed, env_offset=off, **kw)
    orc = CombinatorialOracle(n_envs=B, source=PhiloxSource(B, seed, env_offset=off), **kw)
    R, rows, dims = env.obs_layout
    env.reset()
    orc.reset()
    obs = torch.zeros((T, R, B), device=cuda_device)
    rew = torch.zeros((T, B), dtype=torch.int32, device=cuda_device)
    before = L.launch_count()
    assert env.run_random_access(tp, T, out_obs=obs, obs_stride=R * B, out_reward=rew, reward_stride=B) == T
    assert L.launch_count() - before == 1
    obs, rew = to_np(obs), to_np(rew)
    envs = np.arange(B) + off
    for t in range(1, T + 1):
        tc = orc.source.ctr_t(t)
        a = np.stack([px.lanes16(seed, envs, tc, k, px.PURPOSE_POLICY, C) < px.thr16(tp) for k in range(N)], axis=1)
        o_obs, _, o_rew, o_done, _ = orc.step(a)
        for k in range(N):
            assert np.array_equal(obs[t - 1, rows[k]:rows[k] + dims[k]].T, o_obs[k]), (t, k)
        assert np.array_equal(rew[t - 1], o_rew[:, 0]), t
    assert o_done and to_np(env.done_tensor).all()
    assert np.array_equal(to_np(env.current_buffers), orc.buffers)
    assert np.array_equal(to_np(env.discarded_packets), orc.discarded)
    assert np.array_equal(to_np(env.received_packets), orc.received)
    assert np.array_equal(to_np(env.channel_state), orc.channel_state)
