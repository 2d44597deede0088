"""Independent PPO: one actor and one critic per device (drop-in for algorithms/ippo.py:222-441).

Same constructor, ``train`` / ``test`` / ``create_rollouts`` / ``save`` / ``load`` as the reference ``iPPO``; the
rollout of B lockstep envs, the per-agent networks, the lambda-returns and the clipped-surrogate update run as
sm_100a kernels (csrc/learner_api.cu), all N agents per launch.

Reproducibility: with ``d2d_ppo_b200.use_deterministic_algorithms(True)`` a seeded single-GPU run (same build, GPU
model, ``seed``, ``n_envs`` and ``scratch_bytes``) gives bit-identical parameters, Adam moments, losses, scores and
``test`` results; by default the learner's sums use atomics and runs differ in the last bits.
"""
from __future__ import annotations

import torch

from .. import _lib as L
from . import _dist
from ._base import PPOBase
from ._nets import NetSet, returns_emit, returns_stats


class iPPO(PPOBase):
    _NET_SETS = ("policies", "values")

    def __init__(self, env, hidden_size=128, gamma=0.99, policy_lr=1e-3, value_lr=1e-3, device=None, useRNN=False,
                 save_path=None, combinatorial=False, history_len=10, early_stopping=True, *, seed=0, scratch_bytes=0):
        self._setup(env, hidden_size, gamma, policy_lr, value_lr, device, useRNN, save_path, combinatorial,
                    history_len, early_stopping, seed, scratch_bytes)
        # every agent owns a critic of the policy's architecture with one identity output (ippo.py:143,146)
        self.values = NetSet(self.arch, L.OUT_IDENTITY, self.n_agents, self.B, self.obs_dim, self.obs_off,
                             self.obs_rows, self.hidden_size, 1, self.history_len, self.device, value_lr,
                             scratch_bytes, self._gen, inputs_bf16_exact=self.exact_obs)
        self.value_buf = torch.zeros((self.T, self.n_agents, self.B), dtype=torch.float32, device=self.device)

    # ------------------------------------------------------------------ rollout (ippo.py:277-343)
    def create_rollouts(self, num_episodes=None, forced_actions=None):
        """Returns (obs [T+1 blocks, rows, B] view, actions [T, N, B], log_probs [T, N, B], returns [T, N, B],
        values [T, N, B], advantages [T, N, B], scores [B], dones [T] bools) -- device tensors, env-minor."""
        self._check_episodes(num_episodes)

        N, B = self.n_agents, self.B

        def critic(t):    # agent.value_network(history) on the UNPADDED rollout window (ippo.py:305), written in place
            self.values.rollout_step(self.obs_buf, self.lead, t, out=self.value_buf[t].view(1, N, 1, B))
        scores = self._run_episode(L.ACT_SAMPLE, forced_actions, per_step=critic)
        last = _dist.is_last_shard()
        stats = returns_stats(self.reward_buf, self.value_buf, self.gamma, 0.97, last)
        _dist.all_reduce_sum_(stats)
        norm_a, norm_r = self._norm_stats(stats)             # numpy std (ippo.py:100-101) / torch std (:114-115)
        self.adv_buf, self.ret_buf = returns_emit(self.reward_buf, self.value_buf, self.gamma, 0.97, last,
                                                  norm_a, norm_r, getattr(self, "adv_buf", None),
                                                  getattr(self, "ret_buf", None))
        dones = [t == self.T - 1 for t in range(self.T)]
        self._guard_exact_inputs()
        return (self.obs_buf[self.lead:], self.act_buf, self.logp_buf, self.ret_buf, self.value_buf, self.adv_buf,
                scores, dones)

    # ------------------------------------------------------------------ update (ippo.py:194-217, 418-426)
    def update_epoch(self, cliprange=0.1, beta=0.01):
        """One epoch: every agent's policy step, then its critic step.  Returns ([N] policy losses, [N] value
        losses) as host lists."""
        rows = self.rows_global
        dev = self.device
        sums = torch.zeros((self.n_agents, 2), dtype=torch.float64, device=dev)
        self.policies.zero_grad()
        self.policies.policy_grad(self.obs_buf, self.lead, 0, self.T, self.dist_kind, self.act_buf, self.logp_buf,
                                  self.adv_buf, 1, None, 1.0 / rows, cliprange, beta, sums)
        _dist.all_reduce_sum_(self.policies.grads)         # the PPO gradient all-reduce (NCCL over NVLink)
        self.policies.adam()                               # no gradient clipping in ippo.py
        vsum = torch.zeros(self.n_agents, dtype=torch.float64, device=dev)
        self.values.zero_grad()
        self.values.value_grad(self.obs_buf, self.lead, 0, self.T, 1, self.ret_buf, 1, 1.0 / rows, vsum)
        _dist.all_reduce_sum_(self.values.grads)
        self.values.adam()
        _dist.all_reduce_sum_(sums)
        _dist.all_reduce_sum_(vsum)
        ploss = (-(sums[:, 0] / rows) - beta * sums[:, 1] / rows).tolist()
        return ploss, (vsum / rows).tolist()

    def _epoch_losses(self):
        ploss, vloss = self.update_epoch()
        return ploss[-1], vloss[-1]                        # the reference keeps the last agent's losses (:425-426)

    def train(self, num_iter, n_epoch=4, num_episodes=None, test_freq=100, *, checkpoint_path=None, checkpoint_freq=0,
              resume=False):
        """Returns (scores_episode, score_test_list, policy_loss_list, value_loss_list).  checkpoint_freq = k > 0
        writes the training state into checkpoint_path after iterations 0, k, 2k, ...; resume=True continues the
        run stored there (``PPOBase._train``)."""
        return self._train(num_iter, n_epoch, num_episodes, test_freq, checkpoint_path, checkpoint_freq, resume)
