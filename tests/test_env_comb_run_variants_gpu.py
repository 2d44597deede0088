"""comb_run_kernel's instantiations (exact device counts 4, 6, 8 with homogeneous observations, and the general kernel
for every other shape) against one comb_step_kernel launch per step, bit for bit: every N from 1 to 8, deadlines 7 and
14 (8- and 16-byte records), homogeneous and ragged observations, policy thresholds 0, 1 and 0.2, and switch
probabilities of exactly 0 and 1."""
import numpy as np
import pytest

from _helpers import to_np

pytestmark = pytest.mark.gpu


def _kwargs(N, C, D, homog, T):
    rng = np.random.default_rng(N * 1000 + C * 10 + D)
    sw = rng.uniform(0.0, 0.5, (N, C))
    sw[0, 0], sw[-1, -1] = 1.0, 0.0
    kw = dict(n_agents=N, n_channels=C, deadlines=np.array([D if k % 3 != 1 else D - 4 for k in range(N)]),
              lbdas=np.array([0.4] * N), episode_length=T, traffic_model="aperiodic", channel_switch=sw,
              homogeneous_size=homog)
    if N > 1:   # Bernoulli (periodic) and Poisson devices mixed
        kw.update(traffic_model="heterogeneous", period=np.array([3] * N), arrival_probs=np.array([0.5] * N),
                  offsets=np.arange(N) % 3, periodic_devices=[k for k in range(N) if k % 2 == 1])
    return kw


def _run(kw, B, tp, multi, device):
    import torch
    from d2d_ppo_b200 import _lib as L
    from d2d_ppo_b200.envs import CombinatorialEnv
    T = kw["episode_length"]
    L.set_kernel_switch(L.SWITCH_ENV_MULTISTEP, multi)
    try:
        e = CombinatorialEnv(n_envs=B, device=device, seed=5, env_offset=77, **kw)
        R = e.obs_layout[0]
        e.reset()
        n = T + 4                                                             # crosses a reset
        obs = torch.full((n, R, B), -5.0, device=device)
        rew = torch.full((n, B), -7, dtype=torch.int32, device=device)
        assert e.run_random_access(tp, n, auto_reset=True, out_obs=obs, obs_stride=R * B, out_reward=rew,
                                   reward_stride=B) == n
        obs0 = torch.full((R, B), -5.0, device=device)                        # the same block every step
        acc = torch.zeros(B, dtype=torch.int32, device=device)
        assert e.run_random_access(tp, T - 6, out_obs=obs0, out_reward=acc, accumulate=True) == T - 6
        torch.cuda.synchronize()
        return dict(obs=to_np(obs), rew=to_np(rew), obs0=to_np(obs0), acc=to_np(acc),
                    state=[to_np(x) for x in e._export()])
    finally:
        L.set_kernel_switch(L.SWITCH_ENV_MULTISTEP, 1)


def _check(N, C, D, homog, tp, device, B=333):
    kw = _kwargs(N, C, D, homog, 10)
    on, off = _run(kw, B, tp, 1, device), _run(kw, B, tp, 0, device)
    for key in ("obs", "rew", "obs0", "acc"):
        assert np.array_equal(on[key], off[key]), key
    for x, y in zip(on["state"], off["state"]):
        assert np.array_equal(x, y)
    assert (on["obs"] != -5.0).all() and (on["obs0"] != -5.0).all()
    return on


@pytest.mark.parametrize("homog", [True, False])
@pytest.mark.parametrize("D", [7, 14])
@pytest.mark.parametrize("N", list(range(1, 9)))
def test_comb_run_kernel_every_n(N, D, homog, cuda_device):
    _check(N, 8 if N % 2 == 0 else 4, D, homog, 0.2, cuda_device)


@pytest.mark.parametrize("tp", [0.0, 1.0])
@pytest.mark.parametrize("C", [4, 8])
@pytest.mark.parametrize("N,D,homog", [(6, 14, True), (4, 7, True), (3, 14, False), (6, 7, False)])
def test_comb_run_kernel_policy_threshold_edges(N, D, homog, C, tp, cuda_device):
    """tp = 0: no device transmits, so no reward; tp = 1: every device with a packet transmits on every channel."""
    on = _check(N, C, D, homog, tp, cuda_device)
    if tp == 0.0:
        assert (on["rew"] == 0).all()


@pytest.mark.parametrize("B", [40000, 65536])
def test_comb_run_kernel_bench_shape_sizes(B, cuda_device):
    """The bench's shape (N = 6, C = 8, homogeneous D = 14) with a partial last block and with full blocks."""
    _check(6, 8, 14, True, 0.2, cuda_device, B=B)
