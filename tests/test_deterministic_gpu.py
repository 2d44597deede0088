"""Deterministic mode (d2d_set_deterministic): seeded training is bit-reproducible on every BPTT path, within one
process and across processes, and its gradients stay those of autograd and of the default mode."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from _helpers import rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def deterministic():
    import d2d_ppo_b200
    before = d2d_ppo_b200.are_deterministic_algorithms_enabled()
    d2d_ppo_b200.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        d2d_ppo_b200.use_deterministic_algorithms(before)


@pytest.fixture
def fp32_kernels():
    from d2d_ppo_b200 import _lib as L
    before = L.lib().d2d_get_kernel_switch(L.SWITCH_ALL_TC)
    L.set_kernel_switch(L.SWITCH_ALL_TC, False)
    try:
        yield
    finally:
        L.set_kernel_switch(L.SWITCH_ALL_TC, before)


def _c3_env(dev, B, T, seed=3):
    from d2d_ppo_b200 import presets
    from d2d_ppo_b200.envs import CombinatorialEnv
    kw = presets.combinatorial_kwargs("setup_8_channels", load=1 / 3, episode_length=T)
    return CombinatorialEnv(n_envs=B, device=dev, seed=seed, **kw)


def _sel_env(dev, B, T, seed=3):
    from d2d_ppo_b200.envs import ChannelSelectionEnv
    N, C = 4, 4
    return ChannelSelectionEnv(n_agents=N, n_channels=C, deadlines=np.array([5] * N), lbdas=np.array([0.4] * N),
                               period=None, arrival_probs=None, offsets=None, episode_length=T,
                               traffic_model="aperiodic", periodic_devices=[], channel_switch=np.array([0.1] * (C + 1)),
                               n_envs=B, device=dev, seed=seed)


def _nets(agent):
    if hasattr(agent, "network"):
        return [agent.network]
    return [agent.policies, agent.values if hasattr(agent, "values") else agent.critic]


def _run_ppo(algo, make_env, dev, save, hidden=64, L=6, scratch=0, B=256):
    from d2d_ppo_b200.algorithms.d2d_ppo import D2DPPO
    from d2d_ppo_b200.algorithms.ippo import iPPO
    env = make_env(dev, B, 20)
    comb = env.action_kind == "bernoulli_mask"
    kw = dict(hidden_size=hidden, gamma=0.6, policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=comb,
              history_len=L, early_stopping=False, save_path=save, seed=7, scratch_bytes=scratch)
    np.random.seed(5)                     # D2DPPO shuffles its HAPPO agent order with the global numpy RNG
    if algo == "ippo":
        agent = iPPO(env, **kw)
        res = agent.train(num_iter=2, n_epoch=2, num_episodes=B, test_freq=1)
    else:
        agent = D2DPPO(env, beta_entropy=0.01, **kw)
        res = agent.train(num_iter=2, num_episodes=B, n_epoch=2, test_freq=1)
    torch.cuda.synchronize()
    state = [t.clone() for net in _nets(agent) for t in (net.params, net.adam_m, net.adam_v)]
    return state, res


def _assert_same(a, b):
    (sa, ra), (sb, rb) = a, b
    for x, y in zip(sa, sb):
        assert torch.equal(x, y)
    assert len(ra) == len(rb)
    for x, y in zip(ra, rb):
        assert np.array_equal(np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64))


@pytest.mark.parametrize("algo,env_kind,hidden,fp32,scratch", [
    ("ippo", "c3", 64, False, 0),            # tcgen05 window + recomputing BPTT (gru_bptt_tc)
    ("d2dppo", "c3", 64, False, 0),
    ("ippo", "sel", 64, False, 0),           # inputs not bf16-exact: stored-gate BPTT (gru_bwd_tc)
    ("ippo", "c3", 100, False, 0),           # hidden 100: FP32 BPTT
    ("ippo", "c3", 64, True, 0),             # D2D_SWITCH_ALL_TC = 0: FP32 BPTT
    ("ippo", "c3", 64, False, 64 << 20),     # small scratch: several chunks per call
])
def test_ppo_training_is_bit_reproducible(algo, env_kind, hidden, fp32, scratch, deterministic, tmp_path, request,
                                          cuda_device):
    if fp32:
        request.getfixturevalue("fp32_kernels")
    make_env = _c3_env if env_kind == "c3" else _sel_env
    runs = [_run_ppo(algo, make_env, cuda_device, str(tmp_path / f"best{k}.pt"), hidden=hidden, scratch=scratch)
            for k in range(2)]
    assert os.path.exists(tmp_path / "best0.pt")
    _assert_same(*runs)


@pytest.mark.parametrize("hidden", [64, 100])
def test_irdqn_training_is_bit_reproducible(hidden, deterministic, cuda_device):
    from d2d_ppo_b200.algorithms.irdqn import iRDQN

    def run():
        env = _c3_env(cuda_device, 64, 20, seed=2)
        ag = iRDQN(env, history_len=3, replay_start_size=2, replay_buffer_size=10 ** 5, gamma=0.5,
                   update_target_frequency=3, minibatch_size=32, learning_rate=1e-3, early_stopping=False,
                   hidden_size=hidden, seed=4)
        res = ag.train(6, early_stopping=False)
        torch.cuda.synchronize()
        state = [t.clone() for t in (ag.network.params, ag.network.adam_m, ag.network.adam_v, ag.target_params)]
        return state + [torch.stack(ag.losses)], res
    _assert_same(run(), run())


_CHILD = """
import hashlib, sys, torch
sys.path.insert(0, {root!r})
import d2d_ppo_b200
from d2d_ppo_b200 import presets
from d2d_ppo_b200.algorithms.ippo import iPPO
from d2d_ppo_b200.envs import CombinatorialEnv
d2d_ppo_b200.use_deterministic_algorithms(True)
dev = torch.device("cuda", 0)
env = CombinatorialEnv(n_envs=256, device=dev, seed=3,
                       **presets.combinatorial_kwargs("setup_8_channels", load=1 / 3, episode_length=20))
ag = iPPO(env, hidden_size=64, gamma=0.6, policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=True,
          history_len=6, early_stopping=False, seed=7)
ag.train(num_iter=2, n_epoch=2, num_episodes=256, test_freq=10 ** 9)
h = hashlib.sha256()
for net in (ag.policies, ag.values):
    for t in (net.params, net.adam_m, net.adam_v):
        h.update(t.cpu().numpy().tobytes())
print("SHA256", h.hexdigest())
"""


def test_training_is_bit_reproducible_across_processes(cuda_device):
    hashes = []
    for _ in range(2):
        r = subprocess.run([sys.executable, "-c", _CHILD.format(root=ROOT)], capture_output=True, text=True,
                           cwd=ROOT, timeout=600)
        assert r.returncode == 0, r.stderr[-4000:]
        hashes.append([ln for ln in r.stdout.splitlines() if ln.startswith("SHA256")][-1])
    assert hashes[0] == hashes[1]


def _grads(H, Lh, E, T, I, C, exact, dev):
    """Policy (surrogate) and value (MSE) gradients of fresh random nets on random inputs; seeded, so two calls build
    the same nets and data."""
    from d2d_ppo_b200 import _lib as L
    from d2d_ppo_b200.algorithms._nets import NetSet, action_dtype
    N = 3
    torch.manual_seed(H * 1000 + Lh + 7)
    gen = torch.Generator().manual_seed(H * 1000 + Lh)
    obs = torch.randint(-1, 4, (T, N * I, E), generator=gen).float()
    if not exact:
        obs = obs + 0.25 * torch.rand(obs.shape, generator=gen)
    x = torch.cat([torch.zeros(Lh - 1, N * I, E), obs]).to(dev).contiguous()
    acts = torch.randint(0, 1 << C, (T, N, E), generator=gen).to(action_dtype(L.DIST_BERNOULLI, C)).to(dev)
    adv, ret = torch.randn(T, N, E, generator=gen).to(dev), torch.randn(T, N, E, generator=gen).to(dev)
    logp_old = (-C * 0.69 + 0.05 * torch.randn(T, N, E, generator=gen)).to(dev)
    in_dim, in_off = [I] * N, [k * I for k in range(N)]
    pol = NetSet(L.NET_GRU, L.OUT_SIGMOID, N, E, in_dim, in_off, N * I, H, C, Lh, dev, 1e-3, inputs_bf16_exact=exact)
    val = NetSet(L.NET_GRU, L.OUT_IDENTITY, N, E, in_dim, in_off, N * I, H, 1, Lh, dev, 1e-3, inputs_bf16_exact=exact)
    R = E * T
    sums = torch.zeros((N, 2), dtype=torch.float64, device=dev)
    pol.zero_grad()
    pol.policy_grad(x, Lh - 1, 0, T, L.DIST_BERNOULLI, acts, logp_old, adv, 1, None, 1.0 / R, 0.1, 0.01, sums)
    vsum = torch.zeros(N, dtype=torch.float64, device=dev)
    val.zero_grad()
    val.value_grad(x, Lh - 1, 0, T, 1, ret, 1, 1.0 / R, vsum)
    torch.cuda.synchronize()
    return pol.grads.clone(), val.grads.clone(), sums.clone(), vsum.clone()


SHAPES = [(32, 4, 136, 9, 11, 4, True), (64, 6, 300, 5, 30, 8, True), (64, 5, 260, 4, 40, 8, False),
          (32, 3, 77, 6, 9, 4, False)]


@pytest.mark.parametrize("H,Lh,E,T,I,C,exact", SHAPES)
def test_deterministic_gradients_match_autograd_and_default(H, Lh, E, T, I, C, exact, cuda_device):
    import d2d_ppo_b200
    from test_learner_gpu import test_tensor_core_training_path_vs_autograd
    assert not d2d_ppo_b200.are_deterministic_algorithms_enabled()
    ref = _grads(H, Lh, E, T, I, C, exact, cuda_device)
    d2d_ppo_b200.use_deterministic_algorithms(True)
    try:
        test_tensor_core_training_path_vs_autograd(H, Lh, E, T, I, C, exact, cuda_device)   # against autograd
        det = _grads(H, Lh, E, T, I, C, exact, cuda_device)
        again = _grads(H, Lh, E, T, I, C, exact, cuda_device)
    finally:
        d2d_ppo_b200.use_deterministic_algorithms(False)
    for a, b in zip(det, ref):
        assert rel_err(a, b) < 2e-5
    for a, b in zip(det, again):
        assert torch.equal(a, b)


def test_golden_iterations_in_deterministic_mode(deterministic, cuda_device):
    from test_agents_gpu import test_d2dppo_training_iteration, test_ippo_training_iteration
    test_ippo_training_iteration("c3_gru", cuda_device)
    test_d2dppo_training_iteration("c3_gru", cuda_device)


def test_deterministic_launch_counts(cuda_device):
    """Per chunk of a tcgen05-BPTT net, deterministic mode adds one d(gi) slice sum and one loss-sum reduction; the
    returns statistics add one reduction; the clipped Adam step launches as many kernels as before.  Off again, the
    counts are the default's."""
    import d2d_ppo_b200
    from d2d_ppo_b200 import _lib as L
    from d2d_ppo_b200.algorithms.d2d_ppo import D2DPPO
    from d2d_ppo_b200.algorithms.ippo import iPPO
    env = _c3_env(cuda_device, 256, 20)
    kw = dict(hidden_size=64, gamma=0.6, policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=True,
              history_len=6, early_stopping=False, seed=7)
    ag = iPPO(env, **kw)
    np.random.seed(0)
    ag2 = D2DPPO(_c3_env(cuda_device, 256, 20), **kw)

    def counts():
        n0 = L.launch_count()
        ag.create_rollouts(256)
        n1 = L.launch_count()
        ag.update_epoch()
        n2 = L.launch_count()
        ag2.create_rollouts(256)
        n3 = L.launch_count()
        ag2.update_epoch(cycle=np.arange(6))
        n4 = L.launch_count()
        return n1 - n0, n2 - n1, n3 - n2, n4 - n3
    base = counts()
    d2d_ppo_b200.use_deterministic_algorithms(True)
    try:
        det = counts()
    finally:
        d2d_ppo_b200.use_deterministic_algorithms(False)
    assert det[0] == base[0] + 1                 # returns statistics (iPPO: one two-pass scan)
    assert det[1] == base[1] + 2 * 2             # policy + value net, one chunk each: slice sum + loss reduction
    # D2DPPO: returns statistics of the epoch's advantages; GRU policies: slice sum + loss reduction; MLP critic: loss
    # reduction (the clipped Adam steps launch as many kernels in both modes)
    assert det[3] == base[3] + 4
    assert counts() == base
