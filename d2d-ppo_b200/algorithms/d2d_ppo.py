"""D2D-PPO: HAPPO-style sequential policy updates with a central critic (drop-in for algorithms/d2d_ppo.py:219-461).

The sequential chain M <- ratio_i * M (d2d_ppo.py:427-436) uses each agent's PRE-update ratio, and the agents'
networks are disjoint, so all N forward passes run in one launch, the chain is a running product inside the loss
kernel (csrc/learner_pointwise.cuh: ppo_dlogits_kernel), and all N backward passes run in one launch.

Reproducibility: with ``d2d_ppo_b200.use_deterministic_algorithms(True)`` a seeded single-GPU run is bit-identical
from run to run (same build, GPU model, ``seed``, ``n_envs`` and ``scratch_bytes``).  ``train`` shuffles the HAPPO agent
order with the GLOBAL ``np.random``, as the reference does (d2d_ppo.py:421-422): call ``np.random.seed`` before it, as
the reference scripts do, for a repeatable run.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib as L
from . import _dist
from ._base import PPOBase
from ._nets import NetSet, returns_emit, returns_stats


class D2DPPO(PPOBase):
    def __init__(self, env, hidden_size=128, gamma=0.99, policy_lr=1e-3, value_lr=1e-3, beta_entropy=0.01, device=None,
                 useRNN=False, save_path=None, combinatorial=False, history_len=10, early_stopping=True,
                 *, seed=0, scratch_bytes=0):
        self.beta_entropy = beta_entropy
        self._setup(env, hidden_size, gamma, policy_lr, value_lr, device, useRNN, save_path, combinatorial,
                    history_len, early_stopping, seed, scratch_bytes)
        # the value network "at the BS" sees the global state (d2d_ppo.py:264-267): one MLP, N = 1
        self.critic = NetSet(L.NET_MLP, L.OUT_IDENTITY, 1, self.B, [self.state_rows], [0], self.state_rows,
                             self.hidden_size, 1, 1, self.device, value_lr, scratch_bytes, self._gen)
        self.state_buf = torch.zeros((self.T + 1, self.state_rows, self.B), dtype=torch.float32, device=self.device)
        self._np_rng = np.random          # the reference shuffles the cycle with the global numpy RNG (:421-422)

    # ------------------------------------------------------------------ rollout (d2d_ppo.py:279-339)
    def create_rollouts(self, num_episodes=None, forced_actions=None):
        """Returns (obs view, states [T, S, B], actions [T, N, B], log_probs [T, N, B], rewards [T, B],
        returns [T, B], scores [B], dones [T]) -- device tensors, env-minor."""
        self._check_episodes(num_episodes)
        scores = self._run_episode(L.ACT_SAMPLE, forced_actions, state_buf=self.state_buf)
        last = _dist.is_last_shard()
        stats = returns_stats(self.reward_buf, None, self.gamma, 0.97, last, want_adv=False)
        _dist.all_reduce_sum_(stats)
        # discount_rewards on N identical columns, then .mean(1) (d2d_ppo.py:333,339): one column suffices
        self.ret_buf = returns_emit(self.reward_buf, None, self.gamma, 0.97, last, None,
                                    self._norm_stats(stats)[1])[1][:, 0, :]
        dones = [t == self.T - 1 for t in range(self.T)]
        self._guard_exact_inputs()
        return (self.obs_buf[self.lead:], self.state_buf[:self.T], self.act_buf, self.logp_buf, self.reward_buf,
                self.ret_buf, scores, dones)

    # ------------------------------------------------------------------ update (d2d_ppo.py:413-446)
    def update_epoch(self, cycle=None, cliprange=0.1):
        """One epoch for the agent order ``cycle`` (default: a fresh shuffle).  Returns ([N] policy losses in
        cycle order, value loss)."""
        N, T, dev = self.n_agents, self.T, self.device
        rows = self.rows_global
        if cycle is None:
            cycle = np.arange(N)
            self._np_rng.shuffle(cycle)
        cyc = _dist.broadcast_order(cycle, dev)
        # global advantage estimate at the BS with the critic BEFORE this epoch's updates (:425-427)
        values = self.critic.forward(self.state_buf, 0, 0, T, padded=1)[:, :, 0, :].contiguous()   # [T, 1, B]
        last = _dist.is_last_shard()
        stats = returns_stats(self.reward_buf, values, self.gamma, 0.97, last, want_ret=False)
        _dist.all_reduce_sum_(stats)
        M0 = returns_emit(self.reward_buf, values, self.gamma, 0.97, last,
                          self._norm_stats(stats)[0], None)[0][:, 0, :]                 # [T, B]
        sums = torch.zeros((N, 2), dtype=torch.float64, device=dev)
        self.policies.zero_grad()
        self.policies.policy_grad(self.obs_buf, self.lead, 0, T, self.dist_kind, self.act_buf, self.logp_buf, M0, 0,
                                  cyc, 1.0 / rows, cliprange, self.beta_entropy, sums)
        _dist.all_reduce_sum_(self.policies.grads)         # the PPO gradient all-reduce (NCCL over NVLink)
        self.policies.adam(max_norm=20.0)                  # clip_grad_norm_(20) on the GLOBAL gradient (:211)
        vsum = torch.zeros(1, dtype=torch.float64, device=dev)
        self.critic.zero_grad()
        self.critic.value_grad(self.state_buf, 0, 0, T, 1, self.ret_buf, 0, 1.0 / rows, vsum)
        _dist.all_reduce_sum_(self.critic.grads)
        self.critic.adam(max_norm=20.0)                    # (:445)
        _dist.all_reduce_sum_(sums)
        _dist.all_reduce_sum_(vsum)
        ploss = -(sums[:, 0] / rows) - self.beta_entropy * sums[:, 1] / rows
        order = cyc.tolist()
        return [ploss[i].item() for i in order], (vsum[0] / rows).item()

    def train(self, num_iter, num_episodes=None, n_epoch=4, test_freq=100):
        scores_episode, score_test_list, policy_loss_list, value_loss_list = [], [], [], []
        for it in range(num_iter):
            scores = self.create_rollouts(num_episodes)[6].tolist()
            scores_episode += scores
            for epoch in range(n_epoch):
                ploss_agents, vloss = self.update_epoch()
                policy_loss_list.append(ploss_agents)
                value_loss_list.append(vloss)
                if self._maybe_test(it, epoch, test_freq, scores, score_test_list):
                    return scores_episode, score_test_list, policy_loss_list, value_loss_list
        return scores_episode, score_test_list, policy_loss_list, value_loss_list
