"""Record what every learner entry point launches, to compare two builds of libd2d_b200.so call for call.

For each net of a matrix (MLP / GRU, hidden 16 ... 100, 1 / 5 / 16 outputs, the two-layer Q head, tensor-core kernels
on / off, deterministic mode on / off, n_envs a multiple of 4 or not, exact or inexact inputs, one scratch budget that
fits the call and one that forces one-block chunks) this calls forward, rollout_step, rollout_act, policy_grad
(Bernoulli and categorical), value_grad (shared and per-agent targets) and q_grad (Huber and MSE).  It writes per call,
from one torch.profiler session per net, the ordered kernels with their grid and block and the memsets and copies.
In deterministic mode it adds a hash of the call's outputs (gradients, loss sums, logits, actions and log-probs), which
are then bit-exact.

    python profiles/learner_launch_trace.py --lib OLD.so --out old.jsonl
    python profiles/learner_launch_trace.py --out new.jsonl        # the in-tree library
    cmp old.jsonl new.jsonl

Two builds that launch the same kernels in the same order, with the same outputs, write identical files.
"""
from __future__ import annotations

import argparse
import hashlib
import itertools
import json
import os
import sys
import tempfile

import torch
from torch.profiler import ProfilerActivity, profile, record_function

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, T, L = 3, 6, 4


def _digest(tensors):
    h = hashlib.sha256()
    for t in tensors:
        h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def _launches(events):
    """Chrome-trace events -> {annotation: ordered [name, grid, block] of the kernels (and [name, bytes] of the memsets
    and copies) launched inside that record_function range}."""
    ranges = [(e["ts"], e["ts"] + e["dur"], e["name"]) for e in events if e.get("cat") == "user_annotation"]
    launched_at = {e["args"]["correlation"]: e["ts"] for e in events
                   if e.get("cat") in ("cuda_runtime", "cuda_driver") and "correlation" in e.get("args", {})}
    out = {name: [] for _, _, name in ranges}
    for e in sorted(events, key=lambda e: e.get("ts", 0)):
        cat, a = e.get("cat", ""), e.get("args", {})
        if cat not in ("kernel", "gpu_memset", "gpu_memcpy"):
            continue
        ts = launched_at.get(a.get("correlation"))
        for t0, t1, name in ranges:
            if ts is not None and t0 <= ts <= t1:
                out[name].append([e["name"], a.get("grid"), a.get("block")] if cat == "kernel" else
                                 [e["name"], a.get("bytes")])
    return out


def _inputs(exact, B, rows, gen, dev):
    x = torch.zeros((L - 1 + T, rows, B))
    body = torch.randint(0, 4, (T, rows, B), generator=gen).float() if exact else \
        torch.rand((T, rows, B), generator=gen) * 2 - 1
    x[L - 1:] = body
    return x.to(dev)


def run(lib_path, out_path, quick=False):
    from d2d_ppo_b200 import _lib as Lb
    if lib_path:
        Lb.LIB_PATH = os.path.abspath(lib_path)
    import d2d_ppo_b200
    from d2d_ppo_b200.algorithms._nets import NetSet, action_dtype

    dev = torch.device("cuda", 0)
    tmp = os.path.join(tempfile.mkdtemp(prefix="d2d_trace_"), "trace.json")
    in_dim, in_off, rows = [7, 5, 7], [0, 7, 12], 19
    archs = (("mlp", False), ("gru", True), ("gru", False))
    hidden = (16, 32, 48, 64, 100) if not quick else (32,)
    matrix = list(itertools.product(archs, hidden, (1, 0), (0, 1), (256, 258), (0, 1)))
    n_lines = 0
    with open(out_path, "w") as out:
        for i, ((arch, exact), H, tc, det, B, tiny) in enumerate(matrix):
            O = (1, 5, 16)[i % 3]
            Lb.set_kernel_switch(Lb.SWITCH_ALL_TC, bool(tc))
            d2d_ppo_b200.use_deterministic_algorithms(bool(det))
            gen = torch.Generator().manual_seed(1000 + i)
            a_kind = Lb.NET_GRU if arch == "gru" else Lb.NET_MLP
            lead = L - 1 if arch == "gru" else 0
            x = _inputs(exact, B, rows, gen, dev)[(L - 1 - lead):]
            scratch = 1 if tiny else 0

            def net(out_kind, n_out, head_layers=1):
                return NetSet(a_kind, out_kind, N, B, in_dim, in_off, rows, H, n_out, L, dev, 1e-3,
                              scratch_bytes=scratch, generator=torch.Generator().manual_seed(7 + i),
                              inputs_bf16_exact=exact, head_layers=head_layers)

            cfg = dict(arch=arch, exact=exact, H=H, O=O, tc=tc, det=det, B=B, scratch=scratch)
            calls, hashes = [], {}

            def record(name, fn, outputs):
                torch.cuda.synchronize()
                with record_function(name):
                    fn()
                    torch.cuda.synchronize()
                calls.append(name)
                if det:
                    hashes[name] = _digest(outputs())

            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                w_t = torch.rand((T, B), generator=gen).to(dev) - 0.5
                cyc = torch.arange(N, dtype=torch.int32, device=dev)
                for dist, kind, n_out in ((Lb.DIST_BERNOULLI, Lb.OUT_SIGMOID, O),
                                          (Lb.DIST_CATEGORICAL, Lb.OUT_SOFTMAX, O if O > 1 else 5)):
                    pol = net(kind, n_out)
                    tag = "bernoulli" if dist == Lb.DIST_BERNOULLI else "categorical"
                    if dist == Lb.DIST_BERNOULLI:
                        fwd = {}
                        record("forward", lambda: fwd.setdefault("y", pol.forward(x, lead, 0, T, 1)),
                               lambda: [fwd["y"]])
                        steps = {}
                        record("rollout_step", lambda: steps.update(
                            {t: pol.rollout_step(x, lead, t) for t in range(T)}), lambda: [steps[t] for t in range(T)])
                    dt = action_dtype(dist, n_out)
                    acts = torch.zeros((T, N, B), dtype=dt, device=dev)
                    logp = torch.zeros((T, N, B), device=dev)
                    lg = torch.zeros((T, N, n_out, B), device=dev)

                    def act():
                        for t in range(T):
                            pol.rollout_act(x, lead, t, dist, Lb.ACT_SAMPLE, acts[t], logp[t], seed=11, t_abs0=0,
                                            logits_out=lg[t] if t % 2 else None)
                    record(f"rollout_act_{tag}", act, lambda: [acts, logp, lg])
                    sums = torch.zeros((N, 2), dtype=torch.float64, device=dev)
                    ratio = torch.zeros((T, N, B), device=dev)
                    logp_old = logp + 0.01
                    pol.zero_grad()
                    record(f"policy_grad_{tag}",
                           lambda: pol.policy_grad(x, lead, 0, T, dist, acts, logp_old, w_t, 0, cyc, 1.0 / (T * B),
                                                   0.1, 0.01, sums, ratio),
                           lambda: [pol.grads, sums, ratio])
                    del pol

                val = net(Lb.OUT_IDENTITY, 1)
                for per_agent in (0, 1):
                    tgt = torch.rand((T, N, B) if per_agent else (T, B), generator=gen).to(dev)
                    vsum = torch.zeros(N, dtype=torch.float64, device=dev)
                    vout = torch.zeros((T, N, B), device=dev)
                    val.zero_grad()
                    record(f"value_grad_{'per_agent' if per_agent else 'shared'}",
                           lambda: val.value_grad(x, lead, 0, T, 1, tgt, per_agent, 1.0 / (T * B), vsum, vout),
                           lambda: [val.grads, vsum, vout])
                del val

                q = net(Lb.OUT_IDENTITY, O, head_layers=2 if arch == "gru" else 1)
                qa = torch.randint(0, O, (T, N, B), generator=gen, dtype=torch.uint8).to(dev)
                qt = torch.rand((T, N, B), generator=gen).to(dev)
                for loss_kind, tag in ((Lb.QLOSS_HUBER, "huber"), (Lb.QLOSS_MSE, "mse")):
                    qsum = torch.zeros(N, dtype=torch.float64, device=dev)
                    qout = torch.zeros((T, N, B), device=dev)
                    q.zero_grad()
                    record(f"q_grad_{tag}",
                           lambda: q.q_grad(x, lead, 0, T, qa, qt, loss_kind, 1.0 / (T * B), qsum, qout),
                           lambda: [q.grads, qsum, qout])
                del q
            prof.export_chrome_trace(tmp)
            with open(tmp) as f:
                launches = _launches(json.load(f)["traceEvents"])
            for name in calls:
                assert launches[name], f"{cfg} {name}: no device activity recorded"
                line = dict(cfg, call=name, launches=launches[name])
                if det:
                    line["hash"] = hashes[name]
                out.write(json.dumps(line, sort_keys=True) + "\n")
            n_lines += len(calls)
            torch.cuda.synchronize()
    Lb.set_kernel_switch(Lb.SWITCH_ALL_TC, True)
    d2d_ppo_b200.use_deterministic_algorithms(False)
    print(f"{out_path}: {len(matrix)} nets, {n_lines} calls")


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--lib", default=None, help="libd2d_b200.so to load instead of the in-tree build")
    ap.add_argument("--out", required=True, help="JSON-lines record to write")
    ap.add_argument("--quick", action="store_true", help="hidden size 32 only")
    args = ap.parse_args()
    run(args.lib, args.out, args.quick)
