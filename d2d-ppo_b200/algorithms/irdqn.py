"""Independent recurrent DQN: one GRU Q-network + target network per device (drop-in for algorithms/irdqn.py).

Same constructor arguments, ``train`` / ``test`` return values and quirks as the reference ``iRDQN`` (random
exploration draws only channels {0, 1}, irdqn.py:154; epsilon is a function of the EPISODE index, :253; training
starts after ``replay_start_size`` EPISODES, :233; replay chunks may straddle an episode end, :24-35).  B lockstep envs
each run one episode per iteration of ``train`` (B plays the role of B sequential reference episodes, as in the PPO
learners); every env column keeps its own transition deque inside one device-resident ring, all N agents' networks
run in one launch (net sets with ``head_layers = 2``), and action selection, TD target, loss gradient and the replay
gather are kernels of csrc/dqn_pointwise.cuh.  No step of the path runs in eager PyTorch.

Reproducibility: with ``d2d_ppo_b200.use_deterministic_algorithms(True)`` a seeded single-GPU run (same build, GPU
model, ``seed``, ``n_envs`` and ``scratch_bytes``) is bit-identical from run to run; the replay sampling draws from its
own seeded generator.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from .. import _lib as L
from . import _ckpt, _dist
from ._nets import NetSet, q_select, q_td_target

_LOSSES = {"huber": L.QLOSS_HUBER, "mse": L.QLOSS_MSE}


class ReplayBuffer:
    """Device ring of the last ``n_slots`` episodes of every env column (reference ReplayBuffer, irdqn.py:15-48).

    ``buffer_limit`` counts transitions over all env columns, as the reference's deque does for its single env; it is
    rounded down to whole lockstep episodes (at least two, so that a chunk always fits).  ``len()`` is the number of
    transitions stored per env column (the reference's ``len(buffer)`` at B = 1)."""

    def __init__(self, buffer_limit, device, *, n_envs, n_agents, episode_length, obs_rows, seed=0):
        self.buffer_limit, self.device = int(buffer_limit), torch.device(device)
        self.B, self.N, self.T, self.rows = int(n_envs), int(n_agents), int(episode_length), int(obs_rows)
        self.n_slots = max(2, self.buffer_limit // (self.B * self.T))
        dev = self.device
        self.obs = torch.empty((self.n_slots, self.T + 1, self.rows, self.B), dtype=torch.float32, device=dev)
        self.act = torch.empty((self.n_slots, self.T, self.N, self.B), dtype=torch.uint8, device=dev)
        self.rew = torch.empty((self.n_slots, self.T, self.B), dtype=torch.int32, device=dev)
        self._rng = np.random.default_rng(seed)
        self.reset()

    def reset(self):
        self.n_stored, self.head = 0, 0            # head: slot the next episode is written to

    def __len__(self):
        return self.n_stored * self.T

    @property
    def oldest_slot(self):
        return (self.head - self.n_stored) % self.n_slots

    def add_episode(self, obs_blocks, actions, rewards):
        """The T transitions of one lockstep episode: obs_blocks [T + 1, rows, B] (state of transition t = block t,
        state_next = block t + 1), actions u8 [T, N, B] channel indices, rewards i32 [T, B]."""
        s = self.head
        self.obs[s].copy_(obs_blocks)
        self.act[s].copy_(actions)
        self.rew[s].copy_(rewards)
        self.head = (s + 1) % self.n_slots
        self.n_stored = min(self.n_stored + 1, self.n_slots)

    def _filled(self):
        """The filled slots in ring order (oldest first) as at most two contiguous slot ranges."""
        first = self.oldest_slot
        if first + self.n_stored <= self.n_slots:
            return [slice(first, first + self.n_stored)]
        return [slice(first, self.n_slots), slice(0, self.head)]

    def state_dict(self):
        """The ``n_stored`` filled episodes in ring order (CPU tensors), ``head`` and the sampling generator's state."""
        parts = self._filled()
        return {"n_slots": self.n_slots, "n_stored": self.n_stored, "head": self.head,
                "rng": _ckpt.plain(self._rng.bit_generator.state),
                **{k: torch.cat([getattr(self, k)[s].cpu() for s in parts]) for k in ("obs", "act", "rew")}}

    def load_state_dict(self, d):
        if int(d["n_slots"]) != self.n_slots:
            raise ValueError(f"replay buffer: n_slots is {d['n_slots']} in the stored state but {self.n_slots} here")
        if not (0 <= int(d["n_stored"]) <= self.n_slots and 0 <= int(d["head"]) < self.n_slots):
            raise ValueError(f"replay buffer: n_stored {d['n_stored']} / head {d['head']} out of range")
        for k in ("obs", "act", "rew"):
            own, t = getattr(self, k), d[k]
            if tuple(t.shape[1:]) != tuple(own.shape[1:]) or t.shape[0] != int(d["n_stored"]) or t.dtype != own.dtype:
                raise ValueError(f"replay buffer: {k} is {t.dtype} {tuple(t.shape)} in the stored state, expected "
                                 f"{own.dtype} [{int(d['n_stored'])}, {', '.join(map(str, own.shape[1:]))}]")
        self.n_stored, self.head = int(d["n_stored"]), int(d["head"])
        done = 0
        for s in self._filled():
            n = s.stop - s.start
            for k in ("obs", "act", "rew"):
                getattr(self, k)[s].copy_(d[k][done:done + n])
            done += n
        self._rng.bit_generator.state = d["rng"]

    def sample_chunk(self, batch_size, chunk_size, start_idx=None, env_col=None):
        """``batch_size`` chunks of ``chunk_size`` consecutive transitions (irdqn.py:24-42), gathered on the device.
        start_idx (deque indices, 0 = oldest stored transition of the column) and env_col default to uniform draws as
        in the reference (np.random.randint(0, len - chunk_size)).  Returns env-minor minibatch matrices
        (states [chunk, rows, mb], actions u8 [N, mb], rewards i32 [mb], states_next [chunk, rows, mb], dones u8 [mb]);
        actions / rewards / dones are those of the chunk's LAST transition, the only ones train() uses (:293-296)."""
        mb, dev = int(batch_size), self.device
        if len(self) - chunk_size <= 0:
            raise ValueError(f"replay buffer holds {len(self)} transitions per env: too few for chunks of {chunk_size}")
        if start_idx is None:
            start_idx = self._rng.integers(0, len(self) - chunk_size, mb)
        if env_col is None:
            env_col = self._rng.integers(0, self.B, mb)
        idx = np.stack([np.asarray(start_idx, dtype=np.int32), np.asarray(env_col, dtype=np.int32)])
        if idx.shape != (2, mb) or idx[0].min() < 0 or idx[0].max() + chunk_size > len(self) or \
                idx[1].min() < 0 or idx[1].max() >= self.B:
            raise ValueError("sample_chunk: start_idx / env_col out of range")
        idx = torch.from_numpy(idx).to(dev, non_blocking=True)
        xs = torch.empty((chunk_size, self.rows, mb), dtype=torch.float32, device=dev)
        xn = torch.empty_like(xs)
        act = torch.empty((self.N, mb), dtype=torch.uint8, device=dev)
        rew = torch.empty(mb, dtype=torch.int32, device=dev)
        done = torch.empty(mb, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            L.check(L.lib().d2d_replay_gather(L.ptr(self.obs), L.ptr(self.act), L.ptr(self.rew), L.ptr(idx[0]),
                                              L.ptr(idx[1]), self.oldest_slot, self.n_slots, self.T, int(chunk_size),
                                              self.rows, self.N, self.B, mb, L.ptr(xs), L.ptr(xn), L.ptr(act),
                                              L.ptr(rew), L.ptr(done), L.current_stream()))
        return xs, act, rew, xn, done


class iRDQN:
    def __init__(self, env, history_len=5, replay_start_size=50000, replay_buffer_size=1000000, gamma=0.99,
                 update_target_frequency=10000, minibatch_size=32, learning_rate=1e-3, update_frequency=1,
                 initial_exploration_rate=1, final_exploration_rate=0.1, adam_epsilon=1e-8, loss='huber',
                 early_stopping=True, *, hidden_size=100, seed=0, scratch_bytes=0, device=None):
        if callable(loss) or loss not in _LOSSES:
            raise ValueError("loss must be 'huber' or 'mse' (the loss gradient is a CUDA kernel: no callables)")
        self.device = env.device if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("the learners run on CUDA devices only (no CPU fallback)")
        if getattr(env, "compat", False):
            raise ValueError("construct the env with n_envs=B: the learner rolls out B lockstep episodes per iteration")
        if env.action_kind != "bernoulli_mask":
            raise ValueError("iRDQN steps the env with one-hot channel vectors (irdqn.py:249-257): CombinatorialEnv only")
        self.env = env
        self.history_len = int(history_len)
        self.replay_start_size, self.replay_buffer_size = replay_start_size, replay_buffer_size
        self.gamma = gamma
        self.update_target_frequency, self.update_frequency = update_target_frequency, update_frequency
        self.minibatch_size = int(minibatch_size)
        self.learning_rate, self.adam_epsilon = learning_rate, adam_epsilon
        self.initial_exploration_rate, self.final_exploration_rate = initial_exploration_rate, final_exploration_rate
        self.epsilon = float(initial_exploration_rate)
        self.early_stopping = early_stopping
        self.loss, self._loss_kind = loss, _LOSSES[loss]
        self.hidden_size, self.seed = int(hidden_size), int(seed)
        self.n_agents, self.B, self.T = env.n_agents, env.n_envs, env.episode_length
        self.n_actions = env.action_space[0].n              # irdqn.py:125
        self.n_random = min(2, self.n_actions)              # np.random.randint(0, 2), irdqn.py:154
        self.obs_rows, self.obs_off, self.obs_dim = env.obs_layout
        if len(set(self.obs_dim)) != 1:
            raise ValueError("iRDQN stacks the agents' observations (irdqn.py:236): they must have one size "
                             "(homogeneous_size=True)")
        self.lead = self.history_len - 1
        dev, N, B, T = self.device, self.n_agents, self.B, self.T
        gen = torch.Generator().manual_seed(self.seed)       # identical initial weights on every rank
        common = dict(in_dim=self.obs_dim, in_off=self.obs_off, in_rows=self.obs_rows, hidden=self.hidden_size,
                      n_out=self.n_actions, history_len=self.history_len, device=dev, lr=learning_rate,
                      scratch_bytes=scratch_bytes, inputs_bf16_exact=True, head_layers=2, adam_eps=adam_epsilon)
        # one set of parameters, two kernel handles: minibatch rows for train_step, B rows for act / predict
        self.network = NetSet(L.NET_GRU, L.OUT_IDENTITY, N, self.minibatch_size, generator=gen, **common)
        self.actor = NetSet(L.NET_GRU, L.OUT_IDENTITY, N, B, share_with=self.network, **common)
        self.target_params = self.network.params.clone()     # target_network.load_state_dict(network) (irdqn.py:129)
        self.replay_buffer = ReplayBuffer(replay_buffer_size, dev, n_envs=B, n_agents=N, episode_length=T,
                                          obs_rows=self.obs_rows, seed=self.seed * 7919 + 13 + _dist.rank())
        self._mask_dtype = env._mask_dtype
        self.obs_buf = torch.zeros((self.lead + T + 1, self.obs_rows, B), dtype=torch.float32, device=dev)
        self.act_buf = torch.zeros((T, N, B), dtype=torch.uint8, device=dev)         # channel indices
        self.mask_buf = torch.zeros((T, N, B), dtype=self._mask_dtype, device=dev)   # one-hot action_binary rows
        self.reward_buf = torch.zeros((T, B), dtype=torch.int32, device=dev)
        self.q_buf = torch.zeros((1, N, self.n_actions, B), dtype=torch.float32, device=dev)
        self._loss_sum = torch.zeros(N, dtype=torch.float64, device=dev)
        self._episode = 0
        self.losses = []                                     # per train step: [N] losses (the reference drops them)
        self._progress = self._fresh_progress()
        self._float_lists = _ckpt.FloatLists()

    # ------------------------------------------------------------------ DQN.update_epsilon (irdqn.py:159-161)
    def update_epsilon(self, timestep, horizon_eps=1000):
        eps = self.initial_exploration_rate - \
            (self.initial_exploration_rate - self.final_exploration_rate) * (timestep / horizon_eps)
        self.epsilon = max(eps, self.final_exploration_rate)

    def sync_target(self):
        self.target_params.copy_(self.network.params)

    # ------------------------------------------------------------------ rollout (irdqn.py:231-268, 311-336)
    def _sample_seed(self):
        return (self.seed * 0x9E3779B97F4A7C15 + self._episode * 0xD1B54A32D192ED03 + 0x6A09E667F3BCC909) & (2 ** 64 - 1)

    def _run_episode(self, mode, ready, forced_actions=None, episode=None):
        """One lockstep episode: Q-values of the unpadded history window (irdqn.py:242-247), epsilon-greedy / greedy /
        given channel index per agent, env step with the one-hot channel vectors.  forced_actions: u8 [T, N, B].
        episode: training episode index -- the reference updates every agent's epsilon right after its FIRST action of
        the episode (a.update_epsilon(ep) inside the step loop, :253), so step 0 explores with the previous episode's
        rate and the remaining steps with this episode's."""
        env, N, B = self.env, self.n_agents, self.B
        env.reset_into(self.obs_buf[self.lead])
        for t in range(self.T):
            if forced_actions is not None:
                self.act_buf[t].copy_(forced_actions[t])
                q = None
            else:
                q = self.actor.rollout_step(self.obs_buf, self.lead, t, out=self.q_buf)
            q_select(q, N, B, self.n_actions, L.ACT_GIVEN if forced_actions is not None else mode, self.epsilon, ready,
                     self.n_random, self.act_buf[t], self.mask_buf[t], seed=self._sample_seed(),
                     env_offset=env.env_offset, t_abs=t)
            if t == 0 and episode is not None:
                self.update_epsilon(episode)
            done = env.step_into(self.mask_buf[t], self.obs_buf[self.lead + t + 1], None, self.reward_buf[t])
        assert done
        self._episode += 1

    def _guard_exact_inputs(self):
        """The nets are created with ``inputs_bf16_exact`` (CombinatorialEnv observations are small integers), which lets
        hidden sizes 16 / 32 / 48 / 64 run on the tensor-core GRU window with the observations as ONE bf16 plane.  As in
        the PPO learners the promise is checked on every collected episode, before it enters the replay ring."""
        if self.hidden_size in (16, 32, 48, 64):
            bad = int(self.actor.count_inexact_inputs(self.obs_buf, self.lead, 0, self.T + 1).item())
            if bad:
                raise RuntimeError(f"{bad} observation values are not exactly representable in bf16: the tensor-core "
                                   f"GRU path would truncate them")

    def _packet_sums(self, n=None):
        disc, recv = self.env.discarded_packets, self.env.received_packets        # [B, N]
        n = self.B if n is None else n
        return disc[:n].sum(dtype=torch.float64), recv[:n].sum(dtype=torch.float64)

    # ------------------------------------------------------------------ DQN.train_step (irdqn.py:133-148)
    def train_step(self, transitions):
        """One optimiser step of every agent's network on a sampled minibatch -> [N] losses (device f64)."""
        xs, act, rew, xn, done = transitions
        net, N, mb, Lh = self.network, self.n_agents, self.minibatch_size, self.history_len
        rows = mb * _dist.world_size()
        q_next = net.forward(xn, Lh - 1, 0, 1, 1, params=self.target_params)        # target_network(states_next)
        target = q_td_target(q_next, rew, done, self.gamma)
        net.zero_grad()
        self._loss_sum.zero_()
        net.q_grad(xs, Lh - 1, 0, 1, act.view(1, N, mb), target.view(1, N, mb), self._loss_kind, 1.0 / rows,
                   self._loss_sum)
        _dist.all_reduce_sum_(net.grads)
        net.adam()
        _dist.all_reduce_sum_(self._loss_sum)
        return self._loss_sum / rows

    # ------------------------------------------------------------------ iRDQN.train (irdqn.py:222-302)
    def train(self, n_episodes, early_stopping=True, forced_actions=None, forced_samples=None, *, checkpoint_path=None,
              checkpoint_freq=0, resume=False):
        """``n_episodes`` iterations of B lockstep episodes.  forced_actions(ep) -> u8 [T, N, B] and
        forced_samples(ep) -> (start_idx, env_col) are teacher-forcing hooks of the parity tests.
        Returns (train_scores, test_list, reward_list) like the reference.  checkpoint_freq = k > 0 writes the training
        state into checkpoint_path after episodes 0, k, 2k, ... (their optimiser step and target sync done), after the
        last one and when early stopping fires; resume=True continues the run stored there, if there is one."""
        if (checkpoint_freq or resume) and checkpoint_path is None:
            raise ValueError("checkpoint_freq and resume need a checkpoint_path")
        if resume and _ckpt.exists(checkpoint_path):
            self.load_training_state(checkpoint_path)
        else:
            self._progress = self._fresh_progress()
        p = self._progress
        test_list, reward_list, train_scores = p["test_list"], p["reward_list"], p["train_scores"]
        ep = p["next_episode"]
        while ep < n_episodes and not p["stopped"]:
            ready = ep >= self.replay_start_size
            self._run_episode(L.ACT_SAMPLE, ready, None if forced_actions is None else forced_actions(ep), episode=ep)
            self._guard_exact_inputs()
            self.replay_buffer.add_episode(self.obs_buf[self.lead:], self.act_buf, self.reward_buf)
            train_scores += self.env.compute_urllc().tolist()            # 1 - discarded / received per episode (:272)
            if ep % 100 == 0:
                ts, tr = self.test(50)
                test_list.append(ts)
                reward_list.append(tr)
                if _dist.rank() == 0:
                    print(f"Episode: {ep}, Test score: {ts}, eps: {self.epsilon}, {len(train_scores)}")
                if early_stopping and ts == 1:
                    if _dist.rank() == 0:
                        print(f"Early stopping at episode {ep}")
                    p["stopped"] = True
            if not p["stopped"] and ready and ep % self.update_frequency == 0:
                s = (None, None) if forced_samples is None else forced_samples(ep)
                tr_ = self.replay_buffer.sample_chunk(self.minibatch_size, self.history_len, s[0], s[1])
                self.losses.append(self.train_step(tr_))
                if ep % self.update_target_frequency == 0:
                    self.sync_target()
            p["next_episode"] = ep + 1
            if checkpoint_freq and (ep % checkpoint_freq == 0 or ep + 1 == n_episodes or p["stopped"]):
                self.save_training_state(checkpoint_path)
            ep += 1
        return train_scores, test_list, reward_list

    # ------------------------------------------------------------------ training state (resume an interrupted run)
    @staticmethod
    def _fresh_progress():
        return {"next_episode": 0, "stopped": False, "train_scores": [], "test_list": [], "reward_list": []}

    def save_training_state(self, path):
        """Write everything that decides how ``train`` continues into the directory ``path``: the network with its Adam
        state, the target parameters, epsilon, the episode counters, the loop position, ``losses`` and the lists
        ``train`` returns (rank 0), and every rank's replay shard with its sampling generator.  Call it between
        episodes; the next episode resets the envs.  Collective when a process group is active."""
        p, f = self._progress, self._float_lists
        losses = torch.stack(self.losses).cpu() if self.losses else torch.zeros((0, self.n_agents), dtype=torch.float64)
        replicated = {"network": self.network.training_state(), "target_params": self.target_params.cpu(),
                      "epsilon": float(self.epsilon), "episode": self._episode, "env_episode": self.env.episode,
                      "next_episode": p["next_episode"], "stopped": p["stopped"], "losses": losses,
                      **{k: f.to_tensor(k, p[k]) for k in ("test_list", "reward_list")}}
        local = {"replay": self.replay_buffer.state_dict(),
                 "train_scores": f.to_tensor("train_scores", p["train_scores"])}
        _ckpt.save(path, _ckpt.config(self), replicated, local, self.device)

    def load_training_state(self, path):
        """Restore the state ``save_training_state`` wrote; ValueError if the stored run was set up differently."""
        rep, loc = _ckpt.load(path, _ckpt.config(self))
        self.network.load_training_state(rep["network"])
        if tuple(rep["target_params"].shape) != tuple(self.target_params.shape):
            raise ValueError(f"target_params: expected {tuple(self.target_params.shape)}, got "
                             f"{tuple(rep['target_params'].shape)}")
        self.target_params.copy_(rep["target_params"])
        self.replay_buffer.load_state_dict(loc["replay"])
        self.epsilon, self._episode = float(rep["epsilon"]), int(rep["episode"])
        self.env.set_episode(int(rep["env_episode"]) + 1)
        self.losses = list(rep["losses"].to(self.device).unbind(0))
        f = self._float_lists
        self._progress = {"next_episode": int(rep["next_episode"]), "stopped": bool(rep["stopped"]),
                          "train_scores": f.to_list("train_scores", loc["train_scores"]),
                          **{k: f.to_list(k, rep[k]) for k in ("test_list", "reward_list")}}

    # ------------------------------------------------------------------ iRDQN.test (irdqn.py:305-353)
    def test(self, n_episodes, verbose=False, forced_actions=None):
        """Greedy episodes -> (1 - sum discarded / sum received, mean per-episode sum of mean(max(reward, 0)))."""
        share = _dist.shard(int(n_episodes))[1]
        stats = torch.zeros(4, dtype=torch.float64, device=self.device)
        left = share
        while left > 0:
            n = min(left, self.B)
            self._run_episode(L.ACT_GREEDY, True, forced_actions)
            disc, recv = self._packet_sums(n)
            score = self.reward_buf[:, :n].clamp_min(0).sum(dtype=torch.float64)   # the agents share the reward
            stats += torch.stack([disc, recv, score, torch.tensor(float(n), dtype=torch.float64, device=self.device)])
            left -= n
        _dist.all_reduce_sum_(stats)
        d, r, s, n = stats.tolist()
        return (1 - d / r) if r else float("nan"), s / max(n, 1.0)      # no packet at all: numpy's 0 / 0

    # ------------------------------------------------------------------ checkpoints (not in the reference's iRDQN;
    # same agent_{i}.pth convention as the PPO learners, state_dict keys of irdqn.RNN)
    def save(self, checkpoint_path):
        if _dist.rank() == 0:
            os.makedirs(checkpoint_path, exist_ok=True)
            for i in range(self.n_agents):
                torch.save(self.network.state_dict(i), f"{checkpoint_path}/agent_{i}.pth")

    def load(self, checkpoint_path):
        for i in range(self.n_agents):
            self.network.load_state_dict(i, torch.load(f"{checkpoint_path}/agent_{i}.pth", map_location="cpu"))
        self.sync_target()
