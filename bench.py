#!/usr/bin/env python
"""Headline benchmark: agent-steps/sec of the lockstep env step (+ fused random-access policy).

    python bench.py --gpus N --steps K --warmup W            # this repo, N GPUs (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port), host cores
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's outputs (dump_outputs)

Workload (BASELINE.json configs c3/c5, SURVEY.md section 8d): CombinatorialEnv, setup_8_channels.p, N = 6 devices,
C = 8 channels, deadlines [7,14]x3, heterogeneous traffic at load 1/3, homogeneous_size=True (30 f32 per
observation), 1,048,576 lockstep envs PER GPU (weak scaling; c5's 1M envs on one GPU so the per-step working set,
~1.06 GB, is far larger than the 126 MB L2).  One "step" = one env step of all envs, observations emitted,
actions from the fused CombinatorialRandomAccess policy (algorithms/baselines.py:181-183), reset after every
episode_length = 200 steps inside the timed region.

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_AGENTS, N_CHANNELS, MAX_DEADLINE = 6, 8, 14
OBS_DIM = MAX_DEADLINE + 2 * N_CHANNELS
# Algorithmic bytes per agent-step of the env-step kernel (SURVEY.md section 8d, DESIGN.md section 4):
#   read  buffers D + channel mask 1 + counters 8                      (the action mask is NOT read: fused policy)
#   write buffers D + channel mask 1 + counters 8 + obs 4(D+2C) + (reward 4 + done 1 + ack C) / N
ALG_BYTES = (MAX_DEADLINE + 1 + 8) + (MAX_DEADLINE + 1 + 8 + 4 * OBS_DIM + (5 + N_CHANNELS) / N_AGENTS)
LEAD_IN = 30      # untimed steps enqueued in front of the start event of the timed region (see run_native)
TP = 0.2          # transmission probability of the random-access policy
LOAD = 1 / 3      # xp_load.py:53 first load level
FALLBACK_HBM = 6650.0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--envs", type=int, default=1 << 20, help="lockstep envs per GPU")
    ap.add_argument("--cpu-envs", type=int, default=4096, help="envs per process of the CPU arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-learner-envs", type=int, default=64, help="envs of the CPU iPPO iteration baseline")
    ap.add_argument("--no-configs", action="store_true", help="skip the c1 / c2 / c4 / selection env-step sections")
    ap.add_argument("--no-learner", action="store_true", help="skip the learned-policy rollout / train SPS sections")
    ap.add_argument("--learner-sections", default="rollout,gae,train_c3,train_c3_small,train_c2,irdqn",
                    help="comma list of the learner sections to run (development runs time one section at a time)")
    ap.add_argument("--rollout-envs", type=int, default=65536, help="envs per GPU of the learned-policy rollout (c3)")
    ap.add_argument("--train-envs", type=int, default=65536,
                    help="envs per GPU of the c3 train-SPS sections (BASELINE config 3 names 65,536)")
    ap.add_argument("--train-envs-small", type=int, default=4096, help="extra c3 train-SPS point (round-1 shape)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0's envs) to DIR/<name>.npy, see dump_outputs")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------
# clocks sampled DURING the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi polled every 100 ms.  It is started ~1 s BEFORE the timed region (during untimed spin-up steps
    of the same kernel) because the tool needs several hundred ms to print its first row; only rows whose
    wall-clock arrival falls inside [t_begin, t_end] (the timed region) are summarised when there are any,
    otherwise the rows of the spin-up + timed window are used and `window` says so."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        threading.Thread(target=self._read, daemon=True).start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t_begin=None, t_end=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t_begin is not None and t_begin <= t <= t_end + 0.05]
        window = "timed region"
        if not rows:
            rows, window = [r for (_, r) in self.rows], "spin-up + timed region (timed region shorter than one sample)"
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])), mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's numpy path
# ------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    """Run `steps` env steps (+ random-access policy) of the oracle on `n_envs` envs; returns seconds."""
    n_envs, steps, warmup, seed = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    import numpy as np

    from d2d_ppo_b200 import presets
    from oracle.envs_np import CombinatorialOracle, NumpySource
    kw = presets.combinatorial_kwargs("setup_8_channels", load=LOAD)
    env = CombinatorialOracle(n_envs=n_envs, source=NumpySource(n_envs, seed), **kw)
    rng = np.random.default_rng(seed + 1)
    env.reset()

    def one():
        a = rng.binomial(1, TP, (n_envs, N_AGENTS, N_CHANNELS))      # baselines.py:182
        _, _, _, done, _ = env.step(a)
        if done:
            env.reset()
    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    return time.perf_counter() - t0


def cpu_throughput(n_envs, steps, warmup, procs):
    """agent-steps/s of `procs` independent oracle processes (max time over processes)."""
    if procs == 1:
        dt = _cpu_worker((n_envs, steps, warmup, 0))
    else:
        import multiprocessing as mp
        with mp.get_context("spawn").Pool(procs) as pool:
            dt = max(pool.map(_cpu_worker, [(n_envs, steps, warmup, i) for i in range(procs)]))
    return procs * n_envs * N_AGENTS * steps / dt, dt


def reference_value(cores, episodes):
    """(value, dt, kind, sample) of the reference arm: the UNMODIFIED reference staged in oracle/_ref (one single-env
    instance per host core, CombinatorialRandomAccess.run) when present, else the vectorised oracle port."""
    from d2d_ppo_b200 import presets
    from oracle import make_ref, ref_timing
    if make_ref.verify():
        kw = presets.combinatorial_kwargs("setup_8_channels", load=LOAD)
        v, dt = ref_timing.random_access_throughput(kw, TP, episodes, cores)
        return v, dt, "reference", (
            f"UNMODIFIED reference (oracle/_ref, hashes verified): {cores} processes x 1 env x {episodes} episodes x 200 "
            f"steps of algorithms/baselines.py CombinatorialRandomAccess.run on envs/combinatorial_env.py "
            f"(run_ma_baselines.py:71-74 loop), global np.random, {dt:.1f} s")
    return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    steps, warmup = args.steps, args.warmup
    # bound the sample: one step of 4096 envs costs ~5 ms per process; keep the whole run to ~a minute
    steps_eff = min(steps, 2000)
    port_value, port_dt = cpu_throughput(args.cpu_envs, steps_eff, min(warmup, 50), cores)
    port_sample = (f"{cores} processes x {args.cpu_envs} envs x {steps_eff} steps of oracle/envs_np.CombinatorialOracle "
                   f"(numpy restatement, vectorised over envs) + numpy random-access policy")
    # one reference episode (200 env steps) costs ~25 ms per core: ~20 s per process
    ref = reference_value(cores, episodes=max(4, min(800, 4 * steps_eff // 10)))
    if ref is not None:
        value, dt, kind, sample = ref
    else:
        value, dt, kind, sample = port_value, port_dt, "port", port_sample
    line = {
        "impl": "reference", "metric": "agent-steps/sec (env step + random-access policy)", "value": value,
        "unit": "agent-steps/s", "n_gpus": args.gpus, "steps": steps_eff, "warmup": min(warmup, 50),
        "ms_per_step": port_dt / steps_eff * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": workload_config(cores if kind == "reference" else args.cpu_envs * cores, cpu=True),
        "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": cores, "kind": kind, "sample": sample,
                         "port_value": port_value, "port_sample": port_sample,
                         "note": "value = the reference's own single-env Python loop on every host core; port_value = "
                                 "the numpy restatement vectorised over 4096 envs per process (a far faster CPU "
                                 "program than the reference, kept as the conservative comparison)"},
        "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(envs_total, cpu=False):
    return {"workload": "c5/c3: CombinatorialEnv setup_8_channels.p (N=6, C=8, deadlines [7,14]x3, heterogeneous "
                        "traffic, load 1/3, homogeneous_size=True), fused random-access policy tp=0.2, "
                        "obs f32 emitted, reset every 200 steps",
            "envs_total": envs_total, "n_agents": N_AGENTS, "n_channels": N_CHANNELS, "episode_length": 200,
            "rng": "numpy Generator" if cpu else "philox4x32-10",
            "l2": "n/a" if cpu else "per-step working set ~1.06 GB per GPU >> 126 MB L2 (no flush needed)"}


# ------------------------------------------------------------------------------------------------
# learner sections (extra keys of the JSON line): env + learned-policy rollout, PPO train SPS
# ------------------------------------------------------------------------------------------------
FFMA_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12     # 148 SMs x 128 FP32 FMA lanes x 2 flop x 1.965 GHz = 74.4
FALLBACK_BF16 = 1500.0


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        j = json.load(open(path))
        global BF16_SUSTAINED
        BF16_SUSTAINED = float(j.get("bf16_tflops_sustained", j["bf16_tflops"]))
        return float(j["hbm_gbs"]), float(j["bf16_tflops"]), "of measured (MEASURED_PEAKS.json)"
    return FALLBACK_HBM, FALLBACK_BF16, "of fallback (B200_PROFILING.md)"


BF16_SUSTAINED = FALLBACK_BF16


def gru_tc_issued_flops(I_pad, H, L, head=True):
    """fp16 tensor-pipe flops the fused GRU-window kernel ISSUES per row (csrc/gru_tc.cuh): every fp32 operand is two
    fp16 planes and a product keeps 3 plane pairs.  Per step: h (2 planes) x W_hh (2 planes) as 3 N = 3H MMA groups of
    K = H; x (exact in one plane) x W_ih (2 planes) as 2 N = 4H groups of K = I_pad ([r; z; 0; n] rows).  The fused head
    adds 3 N = H groups of K = H once per row."""
    return 2 * L * (3 * H * 3 * H + 2 * 4 * H * I_pad) + (3 * 2 * H * H if head else 0)


def gru_bptt_issued_flops(I_pad, H, L):
    """fp16 MMA flops of the recomputing BPTT kernel per row (csrc/gru_bptt_tc.cuh): per step the gate recompute
    (as a forward step), D = G W_hh (3 plane pairs, K = 3H, N = H) and dW += G^T P (pairs g0 p0, g1 p0 with N = H + 16,
    g0 p1 with N = H; K = rows, M = 3H counted as the flops of the useful 3H rows)."""
    fwd = 2 * (3 * H * 3 * H + 2 * 4 * H * I_pad)
    return L * (fwd + 2 * 3 * 3 * H * H + 2 * 3 * H * (2 * (H + 16) + H))


def gru_flops_per_agent_step(I, H, L, O):
    """Forward flops of one GRU-window net evaluation as the kernels execute it at rollout time: L input
    projections, L hidden projections, head (SURVEY.md section 8d: 225,792 for I=30, H=64, L=6, O=8)."""
    return 2 * L * 3 * H * (I + H) + 2 * H * H + 2 * H * O


def bench_learner(args, dev, world, rank, barrier, max_over_ranks):
    import numpy as np
    import torch

    from d2d_ppo_b200 import _lib, presets
    from d2d_ppo_b200.algorithms.d2d_ppo import D2DPPO
    from d2d_ppo_b200.algorithms.ippo import iPPO
    from d2d_ppo_b200.envs import CombinatorialEnv, D2DEnv
    out = {}

    def timed(fn):
        barrier()
        n0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) * 1e-3, _lib.launch_count() - n0

    # (ii) env + learned-policy rollout: config c3 = MCA-iPPO of xp_load.py:92-104 (GRU actor + GRU critic per agent,
    #      H = 64, history_len = 6) on the 8-channel combinatorial env, 65,536 lockstep envs per GPU
    B = args.rollout_envs
    kw = presets.combinatorial_kwargs("setup_8_channels", load=LOAD)
    T = kw["episode_length"]
    env = CombinatorialEnv(n_envs=B, device=dev, seed=7, env_offset=rank * B, **kw)
    agent = iPPO(env, hidden_size=64, gamma=0.4, policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=True,
                 history_len=6, early_stopping=False, seed=1, scratch_bytes=6 << 30)
    sections = set(args.learner_sections.split(","))
    agent.create_rollouts(B)                                    # warm-up rollout (scratch allocations, clocks)
    n_roll = 3 if "rollout" in sections else 1
    dt, launches = timed(lambda: [agent.create_rollouts(B) for _ in range(n_roll)])
    dt, launches = dt / n_roll, launches // n_roll
    flops = 2 * gru_flops_per_agent_step(30, 64, 6, 8) - (2 * 64 * 8 - 2 * 64)   # actor (O=8) + critic (O=1)
    steps = world * B * N_AGENTS * T
    hbm_peak, bf16_peak, peak_src = measured_peaks()
    issued = 2 * gru_tc_issued_flops(32, 64, 6)              # actor + critic windows on the tensor pipe
    rollout_entry = {
        "metric": "agent-steps/sec (env step + GRU actor + GRU critic, sampled actions, log-probs, values, "
                  "lambda-returns)", "value": steps / dt, "unit": "agent-steps/s", "envs_per_gpu": B,
        "config": "c3: iPPO useRNN=True hidden 64 history_len 6 on CombinatorialEnv setup_8_channels.p",
        "seconds_per_episode": dt, "gpu_launches": int(launches),
        "roofline": {"bound": "tensor",
                     "note": "primary figure: ALGORITHMIC forward flops (SURVEY.md 8d: 2 L 3H (I + H) + 2 H^2 + 2 H O per "
                             "net, counted once) over the WHOLE rollout time (env step, heads, sampling, returns "
                             "included) against the SUSTAINED bf16 / fp16 peak (a kernel inside a 0.2 s step).  The GRU "
                             "windows run on tcgen05 with fp32 operands split into 2 fp16 planes (fp32 parity at 1e-5), "
                             "i.e. the tensor pipe ISSUES issued_bf16_flops_per_agent_step (3 plane pairs for h W_hh, 2 "
                             "planes of W_ih as N = 4H groups, K padded 30 -> 32, plus the fused head): "
                             "issued_frac_of_sustained is that rate",
                     "achieved": steps / world * flops / dt / 1e12, "peak": BF16_SUSTAINED, "unit": "TFLOP/s",
                     "frac": steps / world * flops / dt / 1e12 / BF16_SUSTAINED, "traffic": None,
                     "flops_per_agent_step": flops, "issued_bf16_flops_per_agent_step": issued,
                     "issued_tflops": steps / world * issued / dt / 1e12,
                     "issued_frac_of_sustained": steps / world * issued / dt / 1e12 / BF16_SUSTAINED,
                     "issued_frac_of_burst": steps / world * issued / dt / 1e12 / bf16_peak,
                     "fp32_ffma_peak_tflops": FFMA_PEAK_TFLOPS,
                     "peak_source": peak_src + " bf16_tflops_sustained"}}

    if "rollout" in sections:
        out["rollout_learned"] = rollout_entry

    # GAE / returns scans of that rollout: lambda-returns + discounted returns for T x N x B elements, two passes
    # (statistics; normalised fp32 emit), HBM-bound.  Algorithmic bytes per element: SURVEY.md section 8d
    from d2d_ppo_b200.algorithms._nets import returns_emit, returns_stats

    def gae_once():
        st = returns_stats(agent.reward_buf, agent.value_buf, 0.4, 0.97, 1)
        na, nr = agent._norm_stats(st)
        returns_emit(agent.reward_buf, agent.value_buf, 0.4, 0.97, 1, na, nr, agent.adv_buf, agent.ret_buf)
    for _ in range(3):
        gae_once()
    reps = 20
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2, rewritten between repetitions
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        flush.fill_(1)
        a.record()
        gae_once()
        b.record()
    torch.cuda.synchronize()
    gae_ms = float(np.median([a.elapsed_time(b) for a, b in evs]))
    elems = T * N_AGENTS * B
    alg = 28 + 5 / N_AGENTS
    moved = 2 * (4 + 4 / N_AGENTS) + 8                                  # what the two passes actually read + write
    gae_entry = {
        "metric": "elements/s of compute_gae + discount_rewards + both normalisations (d2d_ppo.py:100-124)",
        "value": elems / (gae_ms * 1e-3), "unit": "(t, agent, env) elements/s", "elements": elems, "ms": gae_ms,
        "l2": "256 MB flush buffer rewritten before every repetition; working set 0.9 GB",
        "roofline": {"bound": "hbm", "achieved": elems * alg / (gae_ms * 1e-3) / 1e9, "peak": hbm_peak,
                     "unit": "GB/s", "frac": elems * alg / (gae_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                     "alg_bytes_per_element": alg, "moved_bytes_per_element": moved,
                     "moved_gbs": elems * moved / (gae_ms * 1e-3) / 1e9,
                     "note": "algorithmic bytes per SURVEY.md 8d (28 + 5/N: separate scan and normalise passes); the "
                             "kernels recompute the scan in the emit pass instead and move 17.3 B per element, so "
                             "`achieved` may exceed what the DRAM moved; includes the host-side statistics step "
                             "between the two launches", "kernel": "returns_scan_kernel<1>, <2>",
                     "peak_source": peak_src + " hbm_gbs"}}
    del flush
    if "gae" in sections:
        out["gae_returns"] = gae_entry

    del agent, env
    torch.cuda.empty_cache()

    # (iii) PPO train SPS = agent-steps consumed per second of train() (rollout + n_epoch = 5 full-batch updates)
    def train_flops(n_nets_gru, I_pad, H, L, O_list):
        """Per agent-step of ONE update epoch, summed over the GRU nets an agent trains (policy / + critic):
        (algorithmic fp32-equivalent flops, bf16 MMA flops the GRU window + BPTT kernels issue)."""
        alg = issued = 0.0
        for O in O_list:
            fwd = gru_flops_per_agent_step(30, H, L, O)
            alg += 3 * fwd                                               # backward = data + weight gradients = 2 x forward
            issued += gru_tc_issued_flops(I_pad, H, L)                   # forward window + head (training direction)
            issued += gru_bptt_issued_flops(I_pad, H, L)                 # recompute + D = G W_hh + dW += G^T P
        return alg, issued

    def train_sps(make_env, make_agent, B, n_agents, label, n_epoch=5, iters=2, nets=None):
        env = make_env(B)
        ag = make_agent(env)
        kwargs = dict(num_iter=1, n_epoch=n_epoch, num_episodes=B, test_freq=10 ** 9)
        ag._maybe_test = lambda *a, **k: False                   # SPS excludes the periodic evaluation episodes
        ag.train(**kwargs)                                       # warm-up iteration
        kwargs["num_iter"] = iters
        dt, launches = timed(lambda: ag.train(**kwargs))
        # the update alone: one epoch on the rollout in place (device events), for the roofline of the update kernels
        ep_dt, _ = timed(lambda: ag.update_epoch())
        res = {"metric": "PPO train SPS (agent-steps consumed per second of train(): rollout + 5 epochs)",
               "value": world * iters * B * n_agents * env.episode_length / dt, "unit": "agent-steps/s",
               "envs_per_gpu": B, "config": label, "seconds_per_iteration": dt / iters, "gpu_launches": int(launches),
               "seconds_per_epoch": ep_dt}
        if nets is not None:
            alg, issued = train_flops(*nets)
            rows = B * n_agents * env.episode_length
            traffic = None
            tpath = os.path.join(ROOT, "profiles", "train_epoch_traffic.json")
            if os.path.exists(tpath):
                traffic = json.load(open(tpath))
            res["roofline"] = {
                "bound": "tensor", "kernel": "gru_bptt_tc_kernel<64> (+ gru_window_tc_kernel<64,1,*>): ~75 % of an epoch",
                "achieved": rows * alg / ep_dt / 1e12, "peak": BF16_SUSTAINED, "unit": "TFLOP/s",
                "frac": rows * alg / ep_dt / 1e12 / BF16_SUSTAINED,
                "flops_per_agent_step_epoch": alg, "issued_bf16_flops_per_agent_step_epoch": issued,
                "issued_tflops": rows * issued / ep_dt / 1e12,
                "issued_frac_of_sustained": rows * issued / ep_dt / 1e12 / BF16_SUSTAINED,
                "traffic": traffic,
                "note": "one update epoch timed alone with CUDA events; `achieved` = algorithmic fp32-equivalent flops "
                        "of forward + backward of every GRU net (3 x forward), `issued` = fp16 MMA flops of the GRU "
                        "window and BPTT kernels (two fp16 planes per fp32 operand, 3 plane pairs per product, gates "
                        "recomputed in the backward kernel); `traffic` = DRAM bytes per 4,096-env epoch of the two "
                        "dominant kernels from the ncu launch list in profiles/ (null if absent)",
                "peak_source": peak_src + " bf16_tflops_sustained"}
        del ag, env
        torch.cuda.empty_cache()
        return res

    def c3_env(seed):
        return lambda B: CombinatorialEnv(n_envs=B, device=dev, seed=seed, env_offset=rank * B, **kw)

    def c3_ippo(e):
        return iPPO(e, hidden_size=64, gamma=0.4, policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=True,
                    history_len=6, early_stopping=False, seed=2, scratch_bytes=24 << 30)

    def c3_d2dppo(e):
        return D2DPPO(e, hidden_size=64, gamma=0.6, policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=True,
                      history_len=6, early_stopping=False, seed=3, scratch_bytes=24 << 30)

    # BASELINE config 3 names 65,536 envs: that is the headline train figure; the 4,096-env point is kept beside it
    Bt, Bs = args.train_envs, args.train_envs_small
    if "train_c3" not in sections:
        Bt = 0
    if "train_c3_small" not in sections:
        Bs = 0
    if Bt:
        out["train_ippo_c3"] = train_sps(c3_env(8), c3_ippo, Bt, N_AGENTS,
                                         f"c3: iPPO GRU (H 64, L 6) on CombinatorialEnv setup_8_channels.p, {Bt} envs/GPU",
                                         iters=1 if Bt > 16384 else 2, nets=(2, 32, 64, 6, [8, 1]))
        out["train_d2dppo_c3"] = train_sps(c3_env(9), c3_d2dppo, Bt, N_AGENTS,
                                           f"xp_load.py:78-106: D2DPPO GRU (H 64, L 6, gamma .6) on CombinatorialEnv "
                                           f"setup_8_channels.p, {Bt} envs/GPU", iters=1 if Bt > 16384 else 2,
                                           nets=(1, 32, 64, 6, [8]))
    if Bs and Bs != Bt:
        out["train_ippo_c3_small"] = train_sps(c3_env(8), c3_ippo, Bs, N_AGENTS,
                                               f"c3 shape at {Bs} envs/GPU (round-1 bench shape)", nets=(2, 32, 64, 6, [8, 1]))
        out["train_d2dppo_c3_small"] = train_sps(c3_env(9), c3_d2dppo, Bs, N_AGENTS,
                                                 f"xp_load.py shape at {Bs} envs/GPU (round-1 bench shape)",
                                                 nets=(1, 32, 64, 6, [8]))
    if "irdqn" in sections:
        # SURVEY.md 8f-4: independent recurrent DQN with the settings of xp_load.py:112-126 (history_len = n_agents,
        # gamma .4, minibatch 64, lr 1e-4, Huber) on the c3 env; training from iteration 1 on, so every timed iteration
        # is B lockstep epsilon-greedy episodes + the replay-ring copy + one minibatch update of all N Q-networks
        from d2d_ppo_b200.algorithms.irdqn import iRDQN

        def irdqn_sps(B, hidden, iters=3):
            env = CombinatorialEnv(n_envs=B, device=dev, seed=11, env_offset=rank * B, **kw)
            ag = iRDQN(env, history_len=N_AGENTS, replay_start_size=1, replay_buffer_size=100000, gamma=0.4,
                       update_target_frequency=100, minibatch_size=64, learning_rate=1e-4, update_frequency=1,
                       loss="huber", early_stopping=False, hidden_size=hidden, seed=5)
            ag.test = lambda *a, **k: (0.0, 0.0)                 # SPS excludes the periodic evaluation episodes
            import contextlib
            import io
            with contextlib.redirect_stdout(io.StringIO()):      # train() prints a line at every 100th episode
                ag.train(2, early_stopping=False)                 # warm-up: one random and one trained iteration
                ag.replay_start_size = 0
                dt, launches = timed(lambda: ag.train(iters, early_stopping=False))
            return {"metric": "iRDQN train SPS (agent-steps consumed per second of train(): B lockstep "
                              "epsilon-greedy episodes + one minibatch update per iteration)",
                    "value": world * iters * B * N_AGENTS * T / dt, "unit": "agent-steps/s", "envs_per_gpu": B,
                    "config": f"xp_load.py:112-126: iRDQN GRU Q-networks (hidden {hidden}, history_len 6, minibatch 64) "
                              f"on CombinatorialEnv setup_8_channels.p",
                    "seconds_per_iteration": dt / iters, "gpu_launches": int(launches),
                    "kernels": "tcgen05 GRU window + dense head" if hidden in (32, 64) else
                               "FP32 CUDA-core kernels (hidden 100 is the reference's fixed size; the tcgen05 kernels "
                               "take 16 / 32 / 48 / 64)"}
        out["irdqn_c3"] = irdqn_sps(args.train_envs_small, 100)
        out["irdqn_c3_h64"] = irdqn_sps(args.train_envs_small, 64)
    if "train_c2" not in sections:
        return out
    c2 = presets.d2d_c2_kwargs()
    out["train_d2dppo_c2"] = train_sps(
        lambda B: D2DEnv(n_envs=B, device=dev, seed=10, env_offset=rank * B, **c2),
        lambda e: D2DPPO(e, hidden_size=64, gamma=0.6, policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=False,
                         history_len=4, early_stopping=False, seed=4, scratch_bytes=24 << 30),
        4096, 4, "c2: D2DPPO GRU (H 64, L 4) on D2DEnv N=4, 4096 lockstep envs (the named size)")
    return out


# ------------------------------------------------------------------------------------------------
# the other BASELINE configs through the same step kernels (extra key `env_configs`)
# ------------------------------------------------------------------------------------------------
def env_alg_bytes(D, C, N, obs_floats_per_agent, per_env_bytes, action_bytes):
    """SURVEY.md section 8d: (D + m + action + 8) read + (D + m + 8 + 4 obs + per_env / N) written per agent-step,
    m = ceil(C / 8) channel-mask bytes; action_bytes = 0 when the policy is fused into the step kernel."""
    m = (C + 7) // 8
    return (D + m + action_bytes + 8) + (D + m + 8 + 4 * obs_floats_per_agent + per_env_bytes / N)


def bench_env_configs(dev, hbm_peak, steps=200):
    import numpy as np
    import torch

    from d2d_ppo_b200 import presets
    from d2d_ppo_b200.envs import ChannelSelectionEnv, CombinatorialEnv, D2DEnv
    out = []

    def run(label, env, alg, tp=None, actions=None):
        B, N, T = env.n_envs, env.n_agents, env.episode_length
        obs = torch.empty((env.obs_layout[0], B), dtype=torch.float32, device=dev)
        rew = torch.empty(B, dtype=torch.int32, device=dev)

        def one():
            if env.timestep >= T:
                env._reset_device(True, False, out_obs=obs)
            env._step_device(actions, True, False, obs, None, random_access_tp=tp, out_reward=rew)
        env._reset_device(True, False, out_obs=obs)
        for _ in range(5):
            one()
        if tp is not None:
            # the product path of CombinatorialRandomAccess.run: the steps are enqueued by the library in one call
            # (d2d_env_run_random_access); 30 untimed lead-in steps in front of the start event (see run_native)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            env.run_random_access(tp, LEAD_IN, auto_reset=True, out_obs=obs, out_reward=rew)
            e0.record()
            env.run_random_access(tp, steps, auto_reset=True, out_obs=obs, out_reward=rew)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps         # resets (1 in 200 launches) included
        else:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
            ev[0].record()
            for i in range(steps):
                one()
                ev[i + 1].record()
            torch.cuda.synchronize()
            ms = float(np.median([ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]))
        rate = B * N / (ms * 1e-3)
        out.append({"config": label, "envs": B, "n_agents": N, "agent_steps_per_s": rate, "kernel_ms": ms,
                    "alg_bytes_per_agent_step": alg, "achieved_gbs": rate * alg / 1e9,
                    "frac_of_hbm_peak": rate * alg / 1e9 / hbm_peak,
                    "working_set_mb": B * N * alg / 1e6})
        del env, obs
        torch.cuda.empty_cache()

    # c1: run_ma_baselines.py default, 16 channels, ragged observations (deadlines[k] + 2C = 39 / 46 floats)
    kw = presets.combinatorial_kwargs("setup", load=1 / 3, homogeneous_size=False)
    run("c1 CombinatorialEnv setup.p (C=16, ragged obs), fused random access", CombinatorialEnv(
        n_envs=1 << 19, device=dev, seed=1, **kw), env_alg_bytes(10.5, 16, 6, 42.5, 5 + 16, 0), tp=TP)
    # c2: D2DEnv N=4 at the named 4096 envs (L2-resident, launch-latency bound) and at 4M envs (HBM roofline)
    c2 = presets.d2d_c2_kwargs()
    for B in (4096, 1 << 22):
        run(f"c2 D2DEnv N=4 deadlines 7, {B} envs, fused random access", D2DEnv(n_envs=B, device=dev, seed=2, **c2),
            env_alg_bytes(7, 1, 4, 9, 5, 0), tp=TP)
    # c2 through RandomAccess.run's call (rewards accumulated, no observation rows): the steps of an episode run in ONE
    # register-resident kernel (sc_run_kernel; four lanes per env, sc_run_lanes_kernel, up to 32,768 envs); the same call
    # with one launch per step is timed beside it
    from d2d_ppo_b200 import _lib
    for B in (4096, 1 << 22):
        env = D2DEnv(n_envs=B, device=dev, seed=2, **c2)
        acc = torch.zeros(B, dtype=torch.int32, device=dev)
        rates = {}
        for multi in (1, 0):
            _lib.set_kernel_switch(_lib.SWITCH_ENV_MULTISTEP, multi)
            n = 5 * env.episode_length                       # 5 episodes: 5 resets + 5 (or 1000) step launches
            env.run_random_access(TP, env.episode_length, auto_reset=True, out_reward=acc, accumulate=True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            env.run_random_access(TP, n, auto_reset=True, out_reward=acc, accumulate=True)
            e1.record()
            torch.cuda.synchronize()
            rates[multi] = (B * env.n_agents * n / (e0.elapsed_time(e1) * 1e-3), e0.elapsed_time(e1) / n)
        _lib.set_kernel_switch(_lib.SWITCH_ENV_MULTISTEP, 1)
        out.append({"config": f"c2 D2DEnv N=4 deadlines 7, {B} envs, RandomAccess.run (rewards only), multi-step kernel",
                    "envs": B, "n_agents": env.n_agents, "agent_steps_per_s": rates[1][0], "ms_per_step": rates[1][1],
                    "one_launch_per_step_agent_steps_per_s": rates[0][0], "one_launch_per_step_ms": rates[0][1],
                    "bound": "issue (3 Philox calls + update logic per env-step, state in registers)"})
        del env, acc
        torch.cuda.empty_cache()
    # c4: xp_n_agents sweep, C=4, deadlines 7, B x N = 4M
    for N in (4, 16, 64):
        kw = presets.n_agents_sweep_kwargs(N, load=1 / 3)
        run(f"c4 CombinatorialEnv N={N} C=4 aperiodic load 1/3, fused random access", CombinatorialEnv(
            n_envs=(1 << 22) // N, device=dev, seed=3, **kw), env_alg_bytes(7, 4, N, 15, 5 + 4, 0), tp=TP)
    # ChannelSelectionEnv as in xp_gamma.py:43-54 (N=5, C=16): actions from a device tensor (no fused policy)
    N, C = 5, 16
    B = 1 << 20
    sel = ChannelSelectionEnv(n_agents=N, n_channels=C, deadlines=np.array([7] * N), lbdas=np.array([1 / 3] * N),
                              period=None, arrival_probs=None, offsets=None, episode_length=200,
                              traffic_model="aperiodic", periodic_devices=[], channel_switch=np.array([0.2] * (C + 1)),
                              n_envs=B, device=dev, seed=4)
    # global channel state u32 per env (read + written), ack f32 [C+1] per env in the observation only; the fused
    # RandomAccess policy (baselines.py:10-14) reads no action byte
    alg = (7 + 8) + (7 + 8 + 4 * (7 + C + 1)) + (8 + 5 + 4 * (C + 1)) / N
    run("ChannelSelectionEnv xp_gamma.py (N=5, C=16), fused RandomAccess policy", sel, alg, tp=0.0)
    return out


# ------------------------------------------------------------------------------------------------
# native arm
# ------------------------------------------------------------------------------------------------
DUMP_ENVS = 65536     # envs sampled by --dump-outputs: 180 observation rows x 65,536 envs x 4 B = 47 MB


def dump_outputs(directory, env, obs, reward):
    """What a caller of the timed run_random_access call holds after its last step, for a fixed, seeded sample of
    envs: obs [N * OBS_DIM, S] and reward [S] of that step, and the discarded / received packet counters [S, N] the
    URLLC score is computed from, as float32 (every value is exact); env_index [S] float64 names the sampled envs."""
    import numpy as np
    import torch
    idx = np.sort(np.random.default_rng(0).choice(env.n_envs, size=min(env.n_envs, DUMP_ENVS), replace=False))
    sel = torch.from_numpy(idx).to(obs.device)
    out = {"env_index": idx.astype(np.float64),
           "obs": obs.index_select(1, sel).cpu().numpy(),
           "reward": reward.index_select(0, sel).float().cpu().numpy(),
           "discarded": env.discarded_packets.index_select(0, sel).float().cpu().numpy(),
           "received": env.received_packets.index_select(0, sel).float().cpu().numpy()}
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def run_native(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from d2d_ppo_b200 import _lib, presets
    from d2d_ppo_b200.envs import CombinatorialEnv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("for --gpus N > 1 launch with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # host threads and first-touch pinned buffers on the GPU's NUMA node (the e2e leg streams pinned memory)
    from d2d_ppo_b200 import _affinity
    numa = _affinity.bind_to_gpu_numa(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    B, K, W = args.envs, args.steps, args.warmup
    kw = presets.combinatorial_kwargs("setup_8_channels", load=LOAD)
    T = kw["episode_length"]
    # shards are contiguous blocks of the global env index space; no data-path collective (SURVEY.md 8e)
    env = CombinatorialEnv(n_envs=B, device=dev, seed=42, env_offset=rank * B, **kw)
    obs_buf = torch.empty((N_AGENTS * OBS_DIM, B), dtype=torch.float32, device=dev)

    def step():
        if env.timestep >= T:
            env.reset(with_state=False)
        return env.step_random_access(TP, with_state=False, out_obs=obs_buf)

    env.reset(with_state=False)
    for _ in range(max(W, 3)):
        step()

    # ---- device-resident throughput: K steps, CUDA events on the launching stream --------------
    # The K steps (and the resets that fall inside them) are enqueued by ONE call of the C ABI's multi-step entry
    # d2d_env_run_random_access (the library loops over the launches): with a Python -> ctypes call per step, short
    # windows at 8 ranks were bounded by host launch jitter, not by the GPUs (round 1: 0.77 at N = 8, --steps 20).
    rew_buf = torch.zeros(B, dtype=torch.int32, device=dev)

    def run(n):
        done = env.run_random_access(TP, n, auto_reset=True, out_obs=obs_buf, out_reward=rew_buf)
        assert done == n

    sampler = ClockSampler(local)
    sampler.start()
    t_spin = time.perf_counter()
    while time.perf_counter() - t_spin < 1.2:      # untimed spin-up under the same load (see ClockSampler)
        run(50)
        torch.cuda.synchronize()
    # per-launch duration of the step kernel: events between consecutive single-step calls (untimed for the headline)
    n_probe = max(20, min(K, 200))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(n_probe + 1)]
    ev[0].record()
    for i in range(n_probe):
        step()
        ev[i + 1].record()
    torch.cuda.synchronize()
    per = np.array([ev[i].elapsed_time(ev[i + 1]) for i in range(n_probe)])
    kernel_ms = float(np.median(per))             # gaps that contain a reset launch do not move the median
    # the timed steps start from a reset into a fixed episode (Philox streams are keyed by episode and timestep), so
    # their inputs do not depend on how many spin-up steps fitted into the spin-up time
    env.set_episode(0)
    env.reset_into(obs_buf)
    launches0 = _lib.launch_count()
    t_at_start = env.timestep
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.perf_counter()
    # LEAD_IN untimed steps are enqueued IN FRONT of the start event: while the device works through them the host
    # enqueues the K timed launches, so the device-side interval [e0, e1] holds exactly K steps and never waits for the
    # host (a driver-lock hiccup of ~0.5 ms on the first launch after the barrier -- nvidia-smi polls the clocks
    # concurrently -- cost 12 % of a 20-step window at 2 ranks)
    run(LEAD_IN)
    e0.record()
    run(K)
    e1.record()
    host_enqueue_ms = (time.perf_counter() - t_begin) * 1e3
    barrier()
    clocks = sampler.stop(t_begin, time.perf_counter())
    launches_all = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env, obs_buf, rew_buf)
    # launches inside [e0, e1]: the K steps + the resets that fell between them (the lead-in's are not counted)
    t_sim, n_resets = t_at_start, 0
    for i in range(LEAD_IN + K):
        if t_sim >= T:                           # auto_reset: an episode that is over is reset before the step
            t_sim, n_resets = 0, n_resets + (i >= LEAD_IN)
        t_sim += 1
    launches = K + n_resets
    total_ms = max_over_ranks(e0.elapsed_time(e1))
    launch_ms = total_ms / max(launches, 1)       # average launch duration inside the timed region (resets included)
    value = world * B * N_AGENTS * K / (total_ms * 1e-3)

    # ---- end to end through the public API with HOST buffers ------------------------------------
    # env.step_host() = d2d_env_step_host of the C ABI: every step copies that step's actions from pinned host
    # memory (H2D), packs + steps on the device, and copies the step's rewards back into pinned host memory (D2H);
    # the host reads the rewards of step i - 1 after issuing step i (two calls in flight, copies overlap kernels).
    n_host = 4
    rng_host = [np.random.default_rng(i) for i in range(n_host)]
    host_actions = [torch.from_numpy(g.binomial(1, TP, (B, N_AGENTS, N_CHANNELS)).astype(np.uint8)).pin_memory()
                    for g in rng_host]
    w8 = (1 << np.arange(N_CHANNELS)).astype(np.uint8)
    host_masks = [torch.from_numpy(np.ascontiguousarray(((a.numpy() * w8).sum(-1).astype(np.uint8)).T)).pin_memory()
                  for a in host_actions]                                       # device layout: bitmask [N, B]
    host_reward = [torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(2)]
    Ke = max(10, min(K, 200))

    def e2e_run(acts, layout, n):
        checksum, pending = 0, None
        for i in range(n):
            if env.timestep >= T:
                env.reset(with_state=False)
            tk = env.step_host(acts[i % n_host], host_reward[i % 2], layout=layout, with_state=False, out_obs=obs_buf)
            if pending is not None:
                env.host_wait(pending[0])
                checksum += int(pending[1][0]) + int(pending[1][-1])          # the host consumes the result
            pending = (tk, host_reward[i % 2])
        env.host_wait(pending[0])
        return checksum + int(pending[1][0])

    e2e_secs = {}

    def e2e_time(acts, layout):
        e2e_run(acts, layout, 4)
        barrier()
        t0 = time.perf_counter()
        e2e_run(acts, layout, Ke)
        barrier()
        e2e_secs[layout] = max_over_ranks(time.perf_counter() - t0)
        return world * B * N_AGENTS * Ke / e2e_secs[layout]

    # reference layout: with >= 12 host threads the library packs the [B,N,C] bytes to bitmasks on the host before the
    # copy (csrc/host_pack.cpp); the same call with that switched off (device-side packing) is reported beside it
    from d2d_ppo_b200 import _lib as _L
    host_threads = int(_L.lib().d2d_get_host_threads())
    host_packed = host_threads >= 12
    e2e_value = e2e_time(host_actions, "reference")
    secs_default = e2e_secs["reference"]
    pack_state = env.host_pack_state              # 0: the library timed its first calls and fell back to the copy
    host_packed = host_packed and pack_state == 1
    _L.set_kernel_switch(_L.SWITCH_HOST_PACK, False)
    e2e_unpacked = e2e_time(host_actions, "reference")
    secs_unpacked = e2e_secs["reference"]
    _L.set_kernel_switch(_L.SWITCH_HOST_PACK, True)
    e2e_masks = e2e_time(host_masks, "device")
    h2d_step = B * N_AGENTS * (1 if host_packed else N_CHANNELS)
    h2d_gbs_rank = B * N_AGENTS * N_CHANNELS * Ke / secs_unpacked / 1e9

    # ---- roofline of the dominant kernel ---------------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "of measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = FALLBACK_HBM, "of fallback (B200_PROFILING.md 6.65 TB/s)"
    # `achieved`: algorithmic bytes of one launch / the AVERAGE launch duration over the timed region (total time /
    # launches: launch gaps and the cheaper reset launches included, so it can only understate the kernel);
    # kernel_ms = median gap between consecutive single-step launches, reported beside it
    achieved = B * N_AGENTS * ALG_BYTES / (launch_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "env_step_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch")

    # context for the write-heavy mix (83 % of the step kernel's DRAM traffic is stores): what plain fill / copy
    # kernels reach on this GPU right now (torch, 2 GiB buffers, best of 5)
    def _bw(fn, nbytes):
        best = 0.0
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            best = max(best, nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        return best
    scratch_a = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    scratch_b = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    fill_gbs = _bw(lambda: scratch_a.fill_(7), 1 << 30)
    copy_gbs = _bw(lambda: scratch_b.copy_(scratch_a), 2 << 30)
    del scratch_a, scratch_b

    line = {
        "metric": "agent-steps/sec (env step + random-access policy)", "value": value, "unit": "agent-steps/s",
        "n_gpus": world, "steps": K, "warmup": max(W, 3), "ms_per_step": total_ms / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(world * B),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "comb_step_kernel<4,uint8_t,8,1,2>", "kernel_ms": kernel_ms,
                     "avg_launch_ms_timed_region": launch_ms,
                     "achieved_at_median_kernel_ms": B * N_AGENTS * ALG_BYTES / (kernel_ms * 1e-3) / 1e9,
                     "alg_bytes_per_agent_step": ALG_BYTES, "agent_steps_per_launch": B * N_AGENTS,
                     "peak_source": peak_src,
                     "context": {"torch_fill_gbs": fill_gbs, "torch_copy_gbs": copy_gbs,
                                 "note": "write-only and copy bandwidth measured in this run (1 GiB torch fill_ / "
                                         "copy_); the step kernel's traffic is 83 % stores"}},
        "e2e": {"value": e2e_value, "unit": "agent-steps/s",
                "h2d_bytes_per_step": h2d_step, "d2h_bytes_per_step": B * 4, "steps": Ke,
                "api": "CombinatorialEnv.step_host (C ABI d2d_env_step_host): actions u8 [B,N,C] 0/1, the reference's "
                       "(N,C) array per env, in pinned host memory -> i32 [B] rewards in pinned host memory, read by "
                       "the host every step; two calls in flight",
                "host_packed": host_packed, "host_threads": host_threads, "host_pack_state": pack_state,
                "host_bytes_read_per_step": B * N_AGENTS * N_CHANNELS,
                "host_pack_gbs_per_rank": (B * N_AGENTS * N_CHANNELS * Ke / secs_default / 1e9) if host_packed else None,
                "bound": ("host: the library packs the 48 B of actions per env-step into 6 B of channel bitmasks on "
                          f"{host_threads} host threads (AVX2) before they cross PCIe") if host_packed else
                         "PCIe: 48 B of actions per env-step",
                "unpacked_copy": {"value": e2e_unpacked, "unit": "agent-steps/s",
                                  "h2d_bytes_per_step": B * N_AGENTS * N_CHANNELS,
                                  "api": "the same call with D2D_SWITCH_HOST_PACK = 0: the u8 [B,N,C] bytes cross PCIe "
                                         "as they are and are packed on the device (PCIe bound)"},
                "h2d_gbs_per_rank": h2d_gbs_rank, "h2d_gbs_all_ranks": h2d_gbs_rank * world,
                "numa_binding": None if numa is None else {"node": numa[0], "cpus": numa[1]},
                "limiter": ("the host: packing 50.3 MB of u8 [B,N,C] actions per step and rank into 6.3 MB of "
                            "bitmasks (host memory bandwidth and the pool's fork-join per call); unpacked_copy is the "
                            "PCIe-bound alternative, packed_actions the same call when the caller hands in bitmasks")
                           if host_packed else
                           ("host -> device copy of the u8 [B,N,C] actions (50.3 MB per step and rank) over each GPU's "
                            "PCIe link; with N ranks the N concurrent pinned-memory copies share the host's memory / "
                            "root-complex bandwidth, so the per-rank rate drops as N grows (no collective is "
                            "involved); packed_actions moves 8x fewer bytes through the same call; this rank has too "
                            "few host threads for host-side packing"),
                "packed_actions": {"value": e2e_masks, "unit": "agent-steps/s", "h2d_bytes_per_step": B * N_AGENTS,
                                   "d2h_bytes_per_step": B * 4,
                                   "api": "same call with the device action layout (u8 channel bitmask [N,B])"}},
        "gpu_launches": int(launches), "resets_in_timed_region": n_resets, "clocks": clocks,
        "host_enqueue_ms": host_enqueue_ms, "lead_in_steps": LEAD_IN, "launches_incl_lead_in": int(launches_all),
    }
    del obs_buf, env, host_actions, host_masks
    torch.cuda.empty_cache()
    if not args.no_configs:
        line["env_configs"] = bench_env_configs(dev, peak)
    if not args.no_learner:
        line.update(bench_learner(args, dev, world, rank, barrier, max_over_ranks))
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        steps_cpu = 600
        v, dt = cpu_throughput(args.cpu_envs, steps_cpu, 20, 1)
        v1, dt1 = cpu_throughput(1, 3000, 50, 1)
        port = {"value": v, "unit": "agent-steps/s", "cores": 1, "kind": "port",
                "sample": f"{args.cpu_envs} envs x {steps_cpu} steps of oracle/envs_np.CombinatorialOracle (numpy, "
                          f"vectorised over envs) + numpy random-access policy, {dt:.1f} s",
                "single_env_value": v1,
                "single_env_sample": f"1 env x 3000 steps (the reference's own shape: one instance per process), "
                                     f"{dt1:.1f} s"}
        ref = reference_value(1, episodes=400)              # ~10 s of the unmodified reference on one core
        if ref is not None:
            line["cpu_baseline"] = {"value": ref[0], "unit": "agent-steps/s", "cores": 1, "kind": "reference",
                                    "sample": ref[3], "port": port}
        else:
            line["cpu_baseline"] = port
        if not args.no_learner:
            from oracle.ippo_cpu import ippo_iteration_cpu
            threads = torch.get_num_threads()
            r = ippo_iteration_cpu(args.cpu_learner_envs, presets.combinatorial_kwargs("setup_8_channels", load=LOAD),
                                   n_epoch=5)
            from oracle import make_ref, ref_timing
            if make_ref.verify():
                rr = ref_timing.ippo_iteration(presets.combinatorial_kwargs("setup_8_channels", load=LOAD),
                                               num_episodes=2, n_epoch=5, threads=threads)
                line["cpu_baseline_learner_reference"] = {
                    "rollout_value": rr["agent_steps"] / rr["rollout_s"], "train_value": rr["agent_steps"] / rr["total_s"],
                    "unit": "agent-steps/s", "cores": rr["threads"], "kind": "reference",
                    "sample": f"UNMODIFIED reference (oracle/_ref): iPPO.create_rollouts(2) then iPPO.train(num_iter=1, "
                              f"n_epoch=5, num_episodes=2) of algorithms/ippo.py, GRU actor + critic per agent (H 64, "
                              f"L 6) on envs/combinatorial_env.py setup_8_channels.p, torch CPU with {rr['threads']} "
                              f"threads: rollout {rr['rollout_s']:.1f} s, train {rr['total_s']:.1f} s"}
                rq = ref_timing.irdqn_episodes(presets.combinatorial_kwargs("setup_8_channels", load=LOAD),
                                               n_episodes=3, threads=threads)
                line["cpu_baseline_irdqn_reference"] = {
                    "train_value": rq["agent_steps"] / rq["total_s"], "unit": "agent-steps/s", "cores": rq["threads"],
                    "kind": "reference",
                    "sample": f"UNMODIFIED reference (oracle/_ref): iRDQN.train(3) of algorithms/irdqn.py with the "
                              f"settings of xp_load.py:112-126 (replay_start_size 1) on envs/combinatorial_env.py "
                              f"setup_8_channels.p, torch CPU with {rq['threads']} threads: {rq['total_s']:.1f} s"}
            line["cpu_baseline_learner"] = {
                "rollout_value": r["agent_steps"] / r["rollout_s"],
                "train_value": r["agent_steps"] / (r["rollout_s"] + r["update_s"]), "unit": "agent-steps/s",
                "cores": threads, "kind": "port",
                "sample": f"one iPPO iteration (c3: GRU actor + critic per agent, H 64, L 6) of "
                          f"oracle/ippo_cpu.ippo_iteration_cpu on {args.cpu_learner_envs} lockstep envs x 200 steps, "
                          f"5 epochs, torch CPU with {threads} threads: rollout {r['rollout_s']:.1f} s, "
                          f"updates {r['update_s']:.1f} s"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_native(a)
