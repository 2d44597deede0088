"""Shared rollout / evaluation / checkpoint logic of the two learners (reference: create_rollouts, test, save,
load in algorithms/d2d_ppo.py:269-383 and algorithms/ippo.py:266-388).

B lockstep envs each running one episode ARE the reference's ``num_episodes = B`` sequential episodes
(SURVEY.md section 7): rollouts live on the device as env-minor matrices [time][row][env], the env kernels write
observations straight into them, and the policy / critic kernels read them in place.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from .. import _lib as L
from . import _ckpt, _dist
from ._nets import NetSet, action_dtype, returns_norm_stats


class PPOBase:
    def _setup(self, env, hidden_size, gamma, policy_lr, value_lr, device, useRNN, save_path, combinatorial,
               history_len, early_stopping, seed, scratch_bytes):
        self.env = env
        self.history_len = int(history_len)
        self.n_agents = env.n_agents
        self.hidden_size = int(hidden_size)
        self.gamma = gamma
        self.policy_lr, self.value_lr = policy_lr, value_lr
        self.early_stopping = early_stopping
        self.useRNN = bool(useRNN)
        self.save_path = save_path
        self.combinatorial = bool(combinatorial)
        self.device = env.device if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("the learners run on CUDA devices only (no CPU fallback)")
        if getattr(env, "compat", False):
            raise ValueError("construct the env with n_envs=B: the learners roll out B lockstep episodes per "
                             "iteration (B plays the role of the reference's num_episodes)")
        kind = env.action_kind
        if combinatorial and kind != "bernoulli_mask":
            raise ValueError("combinatorial=True (Bernoulli per channel) needs a CombinatorialEnv")
        if not combinatorial and kind == "bernoulli_mask":
            raise ValueError("CombinatorialEnv takes MultiBinary actions: use combinatorial=True")
        self.B, self.T = env.n_envs, env.episode_length
        self.arch = L.NET_GRU if self.useRNN else L.NET_MLP
        self.lead = self.history_len - 1 if self.useRNN else 0
        self.dist_kind = L.DIST_BERNOULLI if combinatorial else L.DIST_CATEGORICAL
        # MLP policies always end in softmax (d2d_ppo.py:81); only the GRU switches to sigmoid (:55-58)
        self.policy_out = L.OUT_SIGMOID if (self.useRNN and combinatorial) else L.OUT_SOFTMAX
        self.n_actions = env.action_space[0].n
        self.obs_rows, self.obs_off, self.obs_dim = env.obs_layout
        self.state_rows = env.state_space.shape[0]
        self.seed = int(seed)
        self._gen = torch.Generator().manual_seed(self.seed)      # identical initial weights on every rank
        self._scratch = int(scratch_bytes)
        # integer-valued observations (buffers, channel bits, ack in {-1, 0, 1}) are exact in bf16, which lets the
        # networks' rollout forward run on the tcgen05 GRU-window kernel; the selection env's 1/count acks are not
        self.exact_obs = kind in ("bernoulli_mask", "binary")
        self.policies = NetSet(self.arch, self.policy_out, self.n_agents, self.B, self.obs_dim, self.obs_off,
                               self.obs_rows, self.hidden_size, self.n_actions, self.history_len, self.device,
                               policy_lr, scratch_bytes, self._gen, inputs_bf16_exact=self.exact_obs)
        self._act_dtype = action_dtype(self.dist_kind, self.n_actions)
        self._iter = 0
        self._progress = self._fresh_progress()
        self._float_lists = _ckpt.FloatLists()
        # rows of the global batch (all ranks): shards may be unequal (_dist.shard leaves a remainder)
        rows = torch.tensor([float(self.B * self.T)], dtype=torch.float64, device=self.device)
        self.rows_global = int(_dist.all_reduce_sum_(rows).item())
        # rollout storage, allocated once: observation blocks lead .. lead + T hold times 0 .. T
        self.obs_buf, self.act_buf, self.logp_buf, self.reward_buf = self._new_rollout_storage()
        # test() rolls out into its OWN storage (allocated on first use): the reference's test() keeps local lists
        # (d2d_ppo.py:341-383) and train() calls it between the epochs of an iteration (:450), so it must not touch
        # the rollout the remaining epochs still update on
        self._eval_storage = None

    def _new_rollout_storage(self):
        T, B, N, dev = self.T, self.B, self.n_agents, self.device
        return (torch.zeros((self.lead + T + 1, self.obs_rows, B), dtype=torch.float32, device=dev),
                torch.zeros((T, N, B), dtype=self._act_dtype, device=dev),
                torch.zeros((T, N, B), dtype=torch.float32, device=dev),
                torch.zeros((T, B), dtype=torch.int32, device=dev))

    # ------------------------------------------------------------------ checkpoints (d2d_ppo.py:269-277)
    def save(self, checkpoint_path):
        if _dist.rank() == 0:
            os.makedirs(checkpoint_path, exist_ok=True)
            for i in range(self.n_agents):
                torch.save(self.policies.state_dict(i), f"{checkpoint_path}/agent_{i}.pth")
            print("Models saved!")

    def load(self, checkpoint_path):
        for i in range(self.n_agents):
            self.policies.load_state_dict(i, torch.load(f"{checkpoint_path}/agent_{i}.pth", map_location="cpu"))
        print("Models loaded!")

    # ------------------------------------------------------------------ training state (resume an interrupted run)
    _NET_SETS = ("policies",)          # subclasses add their value network
    _REPLICATED_LISTS = ("score_test_list", "policy_loss_list", "value_loss_list")

    def _extra_state(self):
        return {}

    def _load_extra_state(self, d):
        pass

    def save_training_state(self, path):
        """Write everything that decides how ``train`` continues into the directory ``path``: both net sets with their
        Adam state, the sampling-stream counter, the env's episode counter, the position of the train loop and the
        lists ``train`` returns.  Call it between iterations; the next rollout resets the envs, so their buffers are
        not part of the state.  Collective when a process group is active."""
        p, f = self._progress, self._float_lists
        replicated = {"nets": {k: getattr(self, k).training_state() for k in self._NET_SETS},
                      "iter": self._iter, "env_episode": self.env.episode, "next_iter": p["next_iter"],
                      "stopped": p["stopped"], **{k: f.to_tensor(k, p[k]) for k in self._REPLICATED_LISTS},
                      **self._extra_state()}
        local = {"scores_episode": f.to_tensor("scores_episode", p["scores_episode"])}   # each rank scores its own envs
        _ckpt.save(path, _ckpt.config(self), replicated, local, self.device)

    def load_training_state(self, path):
        """Restore the state ``save_training_state`` wrote; ValueError if the stored run was set up differently."""
        rep, loc = _ckpt.load(path, _ckpt.config(self))
        for k in self._NET_SETS:
            getattr(self, k).load_training_state(rep["nets"][k])
        self._iter = int(rep["iter"])
        self.env.set_episode(int(rep["env_episode"]) + 1)
        self._load_extra_state(rep)
        f = self._float_lists
        self._progress = {"next_iter": int(rep["next_iter"]), "stopped": bool(rep["stopped"]),
                          "scores_episode": f.to_list("scores_episode", loc["scores_episode"]),
                          **{k: f.to_list(k, rep[k]) for k in self._REPLICATED_LISTS}}

    @staticmethod
    def _fresh_progress():
        return {"next_iter": 0, "stopped": False, "scores_episode": [], "score_test_list": [], "policy_loss_list": [],
                "value_loss_list": []}

    # ------------------------------------------------------------------ rollout
    def _sample_seed(self):
        # one Philox stream per (seed, iteration): timestep t and env index key the draws inside an iteration
        return (self.seed * 0x9E3779B97F4A7C15 + self._iter * 0xD1B54A32D192ED03 + 0x2545F4914F6CDD1D) & (2 ** 64 - 1)

    def _act(self, t, mode, storage, forced=None):
        """select_action for all agents at time t: actions into act_buf[t], log-probs into logp_buf[t]."""
        obs_buf, act_buf, logp_buf, _ = storage
        if forced is not None:
            act_buf[t].copy_(forced)
            mode = L.ACT_GIVEN
        self.policies.rollout_act(obs_buf, self.lead, t, self.dist_kind, mode, act_buf[t], logp_buf[t],
                                  seed=self._sample_seed(), env_offset=self.env.env_offset, t_abs0=t)

    def _run_episode(self, mode, forced_actions=None, state_buf=None, per_step=None, storage=None):
        """One lockstep episode of all B envs.  forced_actions: optional [T, N, B] device-layout actions
        (teacher forcing for parity runs).  per_step(t) runs after the policy acted and before the env steps.
        storage: (obs, act, logp, reward) buffers to roll out into; default = the training rollout."""
        env = self.env
        training = storage is None
        if training:
            storage = (self.obs_buf, self.act_buf, self.logp_buf, self.reward_buf)
        obs_buf, act_buf, _, reward_buf = storage
        env.reset_into(obs_buf[self.lead], None if state_buf is None else state_buf[0])
        for t in range(self.T):
            self._act(t, mode, storage, None if forced_actions is None else forced_actions[t])
            if per_step is not None:
                per_step(t)
            done = env.step_into(act_buf[t], obs_buf[self.lead + t + 1],
                                 None if state_buf is None else state_buf[t + 1], reward_buf[t])
        assert done
        if training:
            self._iter += 1                 # a fresh sampling stream per training rollout; test() is greedy
        return env.compute_urllc()          # score per episode: 1 - discarded / received (d2d_ppo.py:329)

    # ------------------------------------------------------------------ evaluation (d2d_ppo.py:341-383)
    def test(self, num_episodes, forced_actions=None):
        """Greedy rollouts of exactly ``num_episodes`` episodes (split over the ranks; a rank runs its share as
        ceil(share / B) lockstep batches and counts only the first ``share`` episodes).  Returns the reference's
        4-tuple: (mean URLLC score, mean Jain index, total channel errors, mean per-episode sum of the
        agent-mean reward).  Rolls out into evaluation-only storage: the training rollout is left untouched."""
        share = _dist.shard(int(num_episodes))[1]
        if self._eval_storage is None:
            self._eval_storage = self._new_rollout_storage()
        reward_buf = self._eval_storage[3]
        dev = self.device
        stats = torch.zeros(5, dtype=torch.float64, device=dev)
        left = share
        while left > 0:
            n = min(left, self.B)
            s = self._run_episode(L.ACT_GREEDY if forced_actions is None else L.ACT_GIVEN, forced_actions,
                                  storage=self._eval_storage)
            ce = self.env.channel_errors
            ce = ce[:n].to(torch.float64).sum() if torch.is_tensor(ce) else \
                torch.tensor(float(ce) * n, dtype=torch.float64, device=dev)
            stats += torch.stack([s[:n].sum(), self.env.compute_jains()[:n].sum(),
                                  reward_buf[:, :n].to(torch.float64).sum(),     # reward.mean() over equal copies
                                  ce, torch.tensor(float(n), dtype=torch.float64, device=dev)])
            left -= n
        _dist.all_reduce_sum_(stats)
        n = max(stats[4].item(), 1.0)
        return stats[0].item() / n, stats[1].item() / n, int(stats[3].item()), stats[2].item() / n

    # ------------------------------------------------------------------ helpers shared by the train loops
    def _norm_stats(self, stats):
        """(lambda-return norm, return norm), each (mean, std, flags), from the all-reduced [n_cols, 4] sums: numpy's
        population std for compute_gae (d2d_ppo.py:108-109), torch's unbiased std for discount_rewards (:121-123); the
        reference normalises only if EVERY column has a positive std.  One launch, no host round trip."""
        return returns_norm_stats(stats, self.rows_global)

    def _guard_exact_inputs(self):
        """The tensor-core GRU window stages observations as ONE bf16 plane, which is exact for the integer-valued
        observations of CombinatorialEnv / D2DEnv (``exact_obs``).  Checked on every collected rollout: a wrong flag
        would silently truncate the inputs to 8 significant bits.  The count is read where the caller synchronises
        anyway (scores.tolist())."""
        if self.exact_obs and self.useRNN:
            bad = int(self.policies.count_inexact_inputs(self.obs_buf, self.lead, 0, self.T + 1).item())
            if bad:
                raise RuntimeError(f"{bad} observation values are not exactly representable in bf16 although the env "
                                   f"declares integer-valued observations: the tensor-core GRU path would truncate them")

    def _check_episodes(self, num_episodes):
        if num_episodes is not None and int(num_episodes) != self.B:
            raise ValueError(f"num_episodes={num_episodes} but the env runs n_envs={self.B} lockstep episodes per "
                             f"rollout; build the env with n_envs=num_episodes")

    def _maybe_test(self, it, epoch, test_freq, scores, score_test_list):
        """The reference's test / best-model / early-stop block, run once per epoch when iter % test_freq == 0
        (d2d_ppo.py:450-459, ippo.py:428-438).  Returns True to stop training."""
        if it % test_freq != 0:
            return False
        score_test, jains, channel_loss, avg_rewards = self.test(50)
        score_test_list.append(score_test)
        if _dist.rank() == 0:
            print(f"Iteration: {it}, Epoch: {epoch}, score rollout: {np.mean(scores)} "
                  f"Score test: {(score_test, jains, channel_loss, avg_rewards)}")
        if np.max(score_test_list) == score_test and self.save_path is not None:
            self.save(self.save_path)
        return bool((score_test == 1) & bool(self.early_stopping))

    def _train(self, num_iter, n_epoch, num_episodes, test_freq, checkpoint_path, checkpoint_freq, resume):
        """The train loop of both learners; ``_epoch_losses`` runs one epoch and returns the (policy, value) loss
        entries the reference appends.  checkpoint_freq = k writes the training state after iterations 0, k, 2k, ... (their
        epochs and tests done), after the last one and when early stopping fires; resume continues from the state in
        checkpoint_path if there is one."""
        if (checkpoint_freq or resume) and checkpoint_path is None:
            raise ValueError("checkpoint_freq and resume need a checkpoint_path")
        if resume and _ckpt.exists(checkpoint_path):
            self.load_training_state(checkpoint_path)
        else:
            self._progress = self._fresh_progress()
        p = self._progress
        it = p["next_iter"]
        while it < num_iter and not p["stopped"]:
            scores = self.create_rollouts(num_episodes)[6].tolist()
            p["scores_episode"] += scores
            for epoch in range(n_epoch):
                ploss, vloss = self._epoch_losses()
                p["policy_loss_list"].append(ploss)
                p["value_loss_list"].append(vloss)
                if self._maybe_test(it, epoch, test_freq, scores, p["score_test_list"]):
                    p["stopped"] = True
                    break
            p["next_iter"] = it + 1
            # after iterations 0, k, 2k, ...: with k = test_freq right after each test iteration, so that a best model
            # its tests saved belongs to the stored run
            if checkpoint_freq and (it % checkpoint_freq == 0 or it + 1 == num_iter or p["stopped"]):
                self.save_training_state(checkpoint_path)
            it += 1
        return p["scores_episode"], p["score_test_list"], p["policy_loss_list"], p["value_loss_list"]
