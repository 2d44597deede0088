"""What a training-state checkpoint costs late in a long run: one save_training_state (and one load_training_state)
against one training iteration, in the same process.

Workloads:
* iPPO, config c3 (CombinatorialEnv setup_8_channels at load 1/3, 200-step episodes, GRU hidden 64, history 6) at
  65,536 envs, 5 epochs per iteration as in xp_load, no test; its lists filled to their size at iteration 2,000 of
  xp_load (131 M episode scores, 10,000 losses each, 100 test scores);
* iRDQN with the settings of the reference's xp_load iRDQN run (history 6, hidden 100, replay_buffer_size 100,000,
  minibatch 64) at 4,096 envs; replay_start_size 0 so that every timed episode also takes its optimiser step, and two
  warm-up episodes fill the ring (100,000 transitions round up to two whole lockstep episodes); its lists filled to
  their size at episode 20,000 (82 M episode scores, 20,000 [N] losses, 200 test scores and rewards).
An iteration is the rollout and the update without the periodic test.  The filled lists hold random floats; a first
save converts them all, then every timed save follows one more iteration's worth of appended values, as in a run
that checkpoints regularly.  Every timed call ends in a device synchronise.  Files go to a temporary directory that
is removed afterwards.
usage: python profiles/resume_overhead.py [--rounds 3]"""
import argparse
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from d2d_ppo_b200 import presets
from d2d_ppo_b200.algorithms.ippo import iPPO
from d2d_ppo_b200.algorithms.irdqn import iRDQN
from d2d_ppo_b200.envs import CombinatorialEnv

p = argparse.ArgumentParser()
p.add_argument("--rounds", type=int, default=3)
args = p.parse_args()

dev = torch.device("cuda", 0)
try:
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    card = torch.cuda.get_device_name(0)
print(f"device: {card}", flush=True)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def bytes_of(path):
    return sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path))


def report(name, agent, step, fill, append, rounds):
    d = tempfile.mkdtemp(prefix="resume_overhead_")
    try:
        step()                                                          # warm-up
        it = [timed(step) for _ in range(rounds)]
        fill()
        first = timed(lambda: agent.save_training_state(d))
        sv = []
        for _ in range(rounds):
            append()
            sv.append(timed(lambda: agent.save_training_state(d)))
        ld = [timed(lambda: agent.load_training_state(d)) for _ in range(rounds)]
        size = bytes_of(d)
    finally:
        shutil.rmtree(d, ignore_errors=True)
    m = {k: float(np.median(v)) for k, v in (("iter", it), ("save", sv), ("load", ld))}
    print(f"{name}: iteration {m['iter']:.3f} s [{min(it):.3f}, {max(it):.3f}]  save {m['save']:.3f} s "
          f"[{min(sv):.3f}, {max(sv):.3f}] ({m['save'] / m['iter']:.1%} of an iteration)  first save {first:.3f} s  "
          f"load {m['load']:.3f} s [{min(ld):.3f}, {max(ld):.3f}]  files {size / 2 ** 20:.1f} MiB", flush=True)


def floats(n):
    return np.random.default_rng(n).random(n).tolist()


kw = presets.combinatorial_kwargs("setup_8_channels", load=1 / 3, episode_length=200)
B = 65536
env = CombinatorialEnv(n_envs=B, device=dev, seed=42, **kw)
ag = iPPO(env, hidden_size=64, gamma=0.4, policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=True,
          history_len=6, early_stopping=False, seed=1, scratch_bytes=6 << 30)
P = ag._progress


def fill_ppo():
    P["scores_episode"] += floats(2000 * B)
    P["policy_loss_list"] += floats(2000 * 5)
    P["value_loss_list"] += floats(2000 * 5)
    P["score_test_list"] += floats(100)
    P["next_iter"] = 2000


def append_ppo():
    P["scores_episode"] += floats(B)
    P["policy_loss_list"] += floats(5)
    P["value_loss_list"] += floats(5)


report(f"iPPO c3 {B} envs x 200 steps, 5 epochs, state at iteration 2000", ag,
       lambda: (ag.create_rollouts(B), [ag.update_epoch() for _ in range(5)]), fill_ppo, append_ppo, args.rounds)
del P
del ag, env
torch.cuda.empty_cache()

B = 4096
s = presets.SETUPS["setup_8_channels"]
env = CombinatorialEnv(n_envs=B, device=dev, seed=42, **presets.combinatorial_kwargs("setup_8_channels", load=1 / 3,
                                                                                     homogeneous_size=True))
dq = iRDQN(env, history_len=s["n_agents"], replay_start_size=0, replay_buffer_size=100000, gamma=0.4,
           update_target_frequency=100, minibatch_size=64, learning_rate=1e-4, update_frequency=1,
           initial_exploration_rate=1, final_exploration_rate=0.1, adam_epsilon=1e-8, loss="huber", seed=0)
dq.test = lambda *a, **k: (0.0, 0.0)     # time the training episode only (train() tests at every 100th)
dq.train(2, early_stopping=False)
rb = dq.replay_buffer
ring = sum(t.numel() * t.element_size() for t in (rb.obs, rb.act, rb.rew))
print(f"iRDQN replay ring: {rb.n_slots} slots x {B} envs x {dq.T} steps, {ring / 2 ** 30:.2f} GiB", flush=True)
loss = dq.losses[-1]


def fill_dqn():
    Q = dq._progress
    Q["train_scores"] += floats(20000 * B)
    Q["test_list"] += floats(200)
    Q["reward_list"] += floats(200)
    Q["next_episode"] = 20000
    dq.losses += [loss.clone() for _ in range(20000)]


def append_dqn():
    dq._progress["train_scores"] += floats(B)
    dq.losses.append(loss.clone())


report(f"iRDQN xp_load settings, {B} envs, state at episode 20000", dq, lambda: dq.train(1, early_stopping=False),
       fill_dqn, append_dqn, args.rounds)
