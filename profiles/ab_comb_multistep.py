"""A/B inside one process: bench.py's headline workload (CombinatorialEnv setup_8_channels at load 1/3, seed 42, the
timed steps starting from a reset into episode 0, auto reset) through d2d_env_run_random_access with the multi-step
kernel switched on (comb_run_kernel, one launch per episode) and off (one comb_step_kernel launch per step), for three
observation forms:
  stride0  every step writes the same [R, B] block (bench.py; 1,048,576 envs, 4,000 steps)
  strided  every step writes its own block, obs_stride = R * B (524,288 envs, 200 steps: 75 GB of observations)
  none     rewards only (CombinatorialRandomAccess.run; 1,048,576 envs, 4,000 steps)
Prints the median and min / max milliseconds per step over the rounds.
usage: python profiles/ab_comb_multistep.py [--rounds 5]"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from d2d_ppo_b200 import _lib as L, presets
from d2d_ppo_b200.envs import CombinatorialEnv

p = argparse.ArgumentParser()
p.add_argument("--rounds", type=int, default=5)
args = p.parse_args()

dev = torch.device("cuda", 0)
TP = 0.2
kw = presets.combinatorial_kwargs("setup_8_channels", load=1 / 3)
try:
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    card = torch.cuda.get_device_name(0)
print(f"device: {card}", flush=True)


def make(B, K, form):
    env = CombinatorialEnv(n_envs=B, device=dev, seed=42, **kw)
    R = env.obs_layout[0]
    obs = None if form == "none" else torch.empty(((K if form == "strided" else 1) * R, B), device=dev)
    stride = R * B if form == "strided" else 0
    rew = torch.zeros(B, dtype=torch.int32, device=dev)
    env.reset(with_state=False)

    def timed():
        env.set_episode(0)
        env.reset(with_state=False)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        assert env.run_random_access(TP, K, auto_reset=True, out_obs=obs, obs_stride=stride, out_reward=rew) == K
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / K

    return env, timed


for form, B, K in (("stride0", 1 << 20, 4000), ("strided", 1 << 19, 200), ("none", 1 << 20, 4000)):
    env, timed = make(B, K, form)
    ms = {0: [], 1: []}
    try:
        for sw in (0, 1):                      # warm-up of both paths
            L.set_kernel_switch(L.SWITCH_ENV_MULTISTEP, sw)
            timed()
        for rnd in range(args.rounds):
            for sw in (0, 1):
                L.set_kernel_switch(L.SWITCH_ENV_MULTISTEP, sw)
                ms[sw].append(timed())
    finally:
        L.set_kernel_switch(L.SWITCH_ENV_MULTISTEP, 1)
    for sw, name in ((0, "per-step launches"), (1, "multi-step kernel")):
        v = np.array(ms[sw])
        print(f"{form:8s} B={B:8d} K={K:5d} {name:18s}: median {np.median(v):.4f} ms/step "
              f"(min {v.min():.4f}, max {v.max():.4f}, {len(v)} rounds)  "
              f"{B * kw['n_agents'] / np.median(v) * 1e3:.3e} agent-steps/s", flush=True)
    print(f"{form:8s} speed-up (median): {np.median(ms[0]) / np.median(ms[1]):.2f}x", flush=True)
    del env, timed
    torch.cuda.empty_cache()
