"""The learners' and the EDF scheduler's random draws, bit for bit against a numpy restatement on oracle.philox_np:
the Philox counter (env, timestep, agent | policy purpose << 16, block), the key, and the integer / float64 transforms
that turn the words into actions."""
import numpy as np
import pytest
import torch

from oracle import philox_np as px

pytestmark = pytest.mark.gpu

SEED, ENV_OFFSET = 0x1234_5678_9ABC_DEF1, 777


def _policy_words(envs, t, agent, blk):
    """The four policy-stream words of (env, t, agent, block) as uint64 arrays."""
    k0, k1 = SEED & 0xFFFFFFFF, SEED >> 32
    return [w.astype(np.uint64) for w in px.philox4x32_10(envs, t, agent | (px.PURPOSE_POLICY << 16), blk, k0, k1)]


def _head(cuda_device, out_kind, dist_kind, logits):
    from d2d_ppo_b200 import _lib as L
    from d2d_ppo_b200.algorithms._nets import policy_head
    n_t, N, O, B = logits.shape
    actions = torch.empty((n_t, N, B), dtype=torch.int16 if O > 8 else torch.uint8, device=cuda_device)
    logp = torch.empty((n_t, N, B), device=cuda_device)
    probs = torch.empty_like(logits)
    policy_head(logits, N, B, O, out_kind, dist_kind, L.ACT_SAMPLE, actions, logp, probs=probs, seed=SEED,
                env_offset=ENV_OFFSET, t_abs0=5)
    return actions.cpu().numpy().astype(np.int64) & ((1 << O) - 1), probs.cpu().numpy().astype(np.float64)


def test_policy_head_bernoulli_draws(cuda_device):
    """A = 12 channels: three Philox calls (blocks 0, 1, 2) of four 32-bit words; channel j is set iff
    word j % 4 of block j / 4 < p_j 2^32, compared in float64."""
    from d2d_ppo_b200 import _lib as L
    n_t, N, A, B = 2, 3, 12, 4099
    g = torch.Generator().manual_seed(1)
    logits = (torch.randn((n_t, N, A, B), generator=g) * 2).to(cuda_device)
    act, p = _head(cuda_device, L.OUT_SIGMOID, L.DIST_BERNOULLI, logits)
    envs = ENV_OFFSET + np.arange(B)
    for t in range(n_t):
        for agent in range(N):
            want = np.zeros(B, dtype=np.int64)
            for blk in range(3):
                words = _policy_words(envs, 5 + t, agent, blk)
                for lane in range(4):
                    j = 4 * blk + lane
                    bit = words[lane].astype(np.float64) < p[t, agent, j] * 4294967296.0
                    want |= bit.astype(np.int64) << j
            assert np.array_equal(act[t, agent], want), (t, agent)


def test_policy_head_categorical_draws(cuda_device):
    """Inverse CDF in float64: u = (word 0 + 0.5) 2^-32 sum(p), the first j with u < p_0 + .. + p_j."""
    from d2d_ppo_b200 import _lib as L
    n_t, N, A, B = 2, 2, 7, 3001
    g = torch.Generator().manual_seed(2)
    logits = (torch.randn((n_t, N, A, B), generator=g) * 1.5).to(cuda_device)
    act, p = _head(cuda_device, L.OUT_SOFTMAX, L.DIST_CATEGORICAL, logits)
    envs = ENV_OFFSET + np.arange(B)
    for t in range(n_t):
        for agent in range(N):
            cdf = np.cumsum(p[t, agent], axis=0)         # sequential float64 sums, as the kernel adds
            u = (_policy_words(envs, 5 + t, agent, 0)[0].astype(np.float64) + 0.5) * (1.0 / 4294967296.0) * cdf[-1]
            below = u[None, :] < cdf
            want = np.where(below.any(0), below.argmax(0), A - 1)
            assert np.array_equal(act[t, agent], want), (t, agent)


def test_q_select_sample_draws(cuda_device):
    """Epsilon-greedy: word 0 gives u = (w0 + 0.5) 2^-32, greedy iff u >= epsilon; otherwise the action is
    floor(w1 n_random / 2^32)."""
    from d2d_ppo_b200 import _lib as L
    from d2d_ppo_b200.algorithms._nets import q_select
    N, O, B, t_abs, eps = 3, 5, 5003, 9, 0.3
    g = torch.Generator().manual_seed(3)
    q = torch.randn((1, N, O, B), generator=g).to(cuda_device)
    action = torch.empty((N, B), dtype=torch.uint8, device=cuda_device)
    q_select(q, N, B, O, L.ACT_SAMPLE, eps, True, O, action, None, seed=SEED, env_offset=ENV_OFFSET, t_abs=t_abs)
    greedy_act = q[0].cpu().numpy().argmax(1)
    envs = ENV_OFFSET + np.arange(B)
    got = action.cpu().numpy()
    for agent in range(N):
        w = _policy_words(envs, t_abs, agent, 0)
        u = (w[0].astype(np.float64) + 0.5) * (1.0 / 4294967296.0)
        rand = (w[1] * np.uint64(O)) >> np.uint64(32)
        want = np.where(u >= np.float64(np.float32(eps)), greedy_act[agent], rand.astype(np.int64))
        assert np.array_equal(got[agent], want), agent
        assert (u < eps).any() and (u >= eps).any()


def test_edf_empty_buffer_draws(cuda_device):
    """Periodic traffic whose offsets are all non-zero: no packet arrives at the reset, so every env takes EDF's
    fallback, device floor(w0 N / 2^32) of the policy call (env, t = 0, policy << 16, episode)."""
    from d2d_ppo_b200.algorithms.baselines import EarliestDeadlineFirstScheduler
    from d2d_ppo_b200.envs import D2DEnv
    N, B = 5, 2053
    env = D2DEnv(n_agents=N, deadlines=np.array([4] * N), lbdas=np.array([0.5] * N), period=6,
                 arrival_probs=np.array([0.9] * N), offsets=np.array([1, 2, 3, 4, 5]), episode_length=8,
                 traffic_model="periodic", channel_switch=0.2, n_envs=B, device=cuda_device, seed=SEED,
                 env_offset=ENV_OFFSET)
    edf = EarliestDeadlineFirstScheduler(env)
    k0, k1 = SEED & 0xFFFFFFFF, SEED >> 32
    envs = ENV_OFFSET + np.arange(B)
    for episode in range(3):
        env.reset()
        assert env.episode == episode
        assert not env.current_buffers.any()
        got = edf.act().cpu().numpy()
        w0 = px.philox4x32_10(envs, 0, px.PURPOSE_POLICY << 16, episode, k0, k1)[0].astype(np.uint64)
        pick = ((w0 * np.uint64(N)) >> np.uint64(32)).astype(np.int64)
        assert np.array_equal(got, (np.arange(N)[:, None] == pick[None, :]).astype(np.uint8)), episode
