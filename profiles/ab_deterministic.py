"""A/B inside one process: the learner's update epoch with the deterministic mode off and on, alternating.

Workloads: config c3 (CombinatorialEnv setup_8_channels at load 1/3, 200-step episodes, GRU hidden 64, history 6) for
iPPO and D2DPPO, at 4,096 envs and at the 65,536 envs bench.py trains on (scratch_bytes 6 GiB as there).  One rollout
per learner, one warm-up epoch per mode, then --rounds epochs per mode alternating; every timed epoch ends in a device
synchronise.  Prints the median and min / max seconds per epoch and, per net, the chunk length and the activation
scratch the library's plan_chunk allocates (learner_api.cu: floats_per_t and the halo), in both modes.
usage: python profiles/ab_deterministic.py [--rounds 5] [--envs 4096,65536]"""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import d2d_ppo_b200
from d2d_ppo_b200 import presets
from d2d_ppo_b200.algorithms.d2d_ppo import D2DPPO
from d2d_ppo_b200.algorithms.ippo import iPPO
from d2d_ppo_b200.envs import CombinatorialEnv

p = argparse.ArgumentParser()
p.add_argument("--rounds", type=int, default=5)
p.add_argument("--envs", default="4096,65536")
args = p.parse_args()

dev = torch.device("cuda", 0)
T, H, LH, SCRATCH = 200, 64, 6, 6 << 30
try:
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    card = torch.cuda.get_device_name(0)
print(f"device: {card}", flush=True)


def scratch(net, det, n_t=T):
    """(chunk length, bytes) of the training scratch plan_chunk sets up for `net` (GRU, tcgen05 BPTT)."""
    NB, L, O = net.N * net.B, net.L, net.O
    per_t = (H + O + 6 * H + L * H + O + H + 5 * H + (L * 3 * H if det else 0)) * NB
    halo = (L - 1) * 3 * H * NB * 2
    tc = max(1, min(n_t, (SCRATCH // 4 - halo) // per_t))
    return tc, 4 * (per_t * tc + halo)


def epoch(agent, algo):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    agent.update_epoch() if algo == "ippo" else agent.update_epoch(cycle=np.arange(agent.n_agents))
    torch.cuda.synchronize()
    return time.perf_counter() - t0


kw = presets.combinatorial_kwargs("setup_8_channels", load=1 / 3, episode_length=T)
for B in [int(b) for b in args.envs.split(",")]:
    for algo in ("ippo", "d2dppo"):
        env = CombinatorialEnv(n_envs=B, device=dev, seed=42, **kw)
        common = dict(hidden_size=H, gamma=0.4, policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=True,
                      history_len=LH, early_stopping=False, seed=1, scratch_bytes=SCRATCH)
        agent = iPPO(env, **common) if algo == "ippo" else D2DPPO(env, **common)
        agent.create_rollouts(B)
        times = {False: [], True: []}
        for det in (False, True):          # warm-up: both modes' kernels loaded, scratch grown
            d2d_ppo_b200.use_deterministic_algorithms(det)
            epoch(agent, algo)
        for _ in range(args.rounds):
            for det in (False, True):
                d2d_ppo_b200.use_deterministic_algorithms(det)
                times[det].append(epoch(agent, algo))
        d2d_ppo_b200.use_deterministic_algorithms(False)
        med = {d: float(np.median(v)) for d, v in times.items()}
        print(f"{algo} c3 {B} envs x {T} steps: update epoch default {med[False]:.4f} s "
              f"[{min(times[False]):.4f}, {max(times[False]):.4f}]  deterministic {med[True]:.4f} s "
              f"[{min(times[True]):.4f}, {max(times[True]):.4f}]  ratio {med[True] / med[False]:.3f}", flush=True)
        nets = [("policy", agent.policies)] + ([("value", agent.values)] if algo == "ippo" else [])
        for name, net in nets:
            (tc0, b0), (tc1, b1) = scratch(net, False), scratch(net, True)
            print(f"  {name} net scratch: default Tc {tc0} ({b0 / 2 ** 30:.2f} GiB), deterministic Tc {tc1} "
                  f"({b1 / 2 ** 30:.2f} GiB)", flush=True)
        del agent, env
        torch.cuda.empty_cache()
