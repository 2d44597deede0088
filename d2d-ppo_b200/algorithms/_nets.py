"""Host-side handles for the learner kernels: parameter buffers, optimiser state, checkpoints.

Plumbing only: PyTorch owns the device memory; every computation is a C-ABI call into libd2d_b200.so
(csrc/learner_api.cu).  A ``NetSet`` is the N per-agent networks the reference builds one ``PPO`` object at a
time (algorithms/d2d_ppo.py:252-262, algorithms/ippo.py:254-264).
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from .. import _lib as L

GRU_KEYS = ["lstm.weight_ih_l0", "lstm.weight_hh_l0", "lstm.bias_ih_l0", "lstm.bias_hh_l0",
            "layers.0.weight", "layers.0.bias", "layers.2.weight", "layers.2.bias"]
MLP_KEYS = ["linear1.weight", "linear1.bias", "linear2.weight", "linear2.bias"]
# the Q-network of algorithms/irdqn.py:58-72: one more hidden Linear + ReLU behind the GRU
GRU_Q_KEYS = GRU_KEYS[:6] + ["layers.2.weight", "layers.2.bias", "layers.4.weight", "layers.4.bias"]


def _orthogonal(rows, cols, gain, generator):
    """torch.nn.init.orthogonal_ (the reference's init_weights, d2d_ppo.py:17-21) on the host."""
    w = torch.empty(rows, cols)
    torch.nn.init.orthogonal_(w, gain, generator=generator)
    return w


class NetSet:
    """N independent networks of one architecture evaluated in one launch (grid.y = agent)."""

    def __init__(self, arch, out_kind, n_agents, n_envs, in_dim, in_off, in_rows, hidden, n_out, history_len, device,
                 lr, scratch_bytes=0, generator=None, inputs_bf16_exact=False, head_layers=1, adam_eps=1e-8,
                 share_with=None):
        """head_layers = 2: the GRU Q-network of irdqn.py.  share_with: another NetSet of the same architecture
        (any n_envs) whose parameter / gradient / optimiser buffers this handle aliases -- the kernels of a handle are
        sized for its n_envs, so a learner that evaluates the same networks on B rollout envs and on a minibatch of
        other size holds two handles over one set of parameters."""
        self.arch, self.out_kind = arch, out_kind
        self.head_layers, self.adam_eps = int(head_layers), float(adam_eps)
        self.N, self.B, self.H, self.O = int(n_agents), int(n_envs), int(hidden), int(n_out)
        self.L = int(history_len) if arch == L.NET_GRU else 1
        self.in_dim = [int(i) for i in in_dim]
        self.in_off = [int(i) for i in in_off]
        self.in_rows = int(in_rows)
        self.device = torch.device(device)
        self.lr = float(lr)
        self._lib = L.lib()
        a_dim = np.asarray(self.in_dim, dtype=np.int32)
        a_off = np.asarray(self.in_off, dtype=np.int32)
        cfg = L.NetConfig(arch=arch, out_kind=out_kind, n_agents=self.N, n_envs=self.B, hidden=self.H, n_out=self.O,
                          history_len=self.L, in_rows=self.in_rows,
                          in_dim=a_dim.ctypes.data_as(C.POINTER(C.c_int32)),
                          in_off=a_off.ctypes.data_as(C.POINTER(C.c_int32)), scratch_bytes=int(scratch_bytes),
                          inputs_bf16_exact=int(bool(inputs_bf16_exact)), head_layers=self.head_layers)
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            L.check(self._lib.d2d_net_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.stride = int(self._lib.d2d_net_param_stride(h))
        self.keys = (GRU_Q_KEYS if self.head_layers == 2 else GRU_KEYS) if arch == L.NET_GRU else MLP_KEYS
        self._layout = []
        for g in range(self.N):
            per = []
            for i in range(len(self.keys)):
                off, rows, cols = C.c_int64(), C.c_int32(), C.c_int32()
                L.check(self._lib.d2d_net_tensor(h, g, i, C.byref(off), C.byref(rows), C.byref(cols)))
                per.append((off.value, rows.value, cols.value))
            self._layout.append(per)
        self._sqnorm = torch.zeros(self.N, dtype=torch.float64, device=self.device)
        self._owner = share_with
        if share_with is not None:
            if (share_with.arch, share_with.N, share_with.stride, share_with.keys) != \
                    (self.arch, self.N, self.stride, self.keys):
                raise ValueError("share_with: the two net sets differ in architecture")
            self.params, self.grads = share_with.params, share_with.grads
            self.adam_m, self.adam_v = share_with.adam_m, share_with.adam_v
            return
        self.params = torch.zeros((self.N, self.stride), dtype=torch.float32, device=self.device)
        self.grads = torch.zeros_like(self.params)
        self.adam_m = torch.zeros_like(self.params)
        self.adam_v = torch.zeros_like(self.params)
        self.adam_step = 0
        self.reset_parameters(generator)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self._lib.d2d_net_destroy(h)
            except Exception:
                pass
            self._h = None

    # ---------------------------------------------------------------- parameters
    def reset_parameters(self, generator=None):
        """The reference's initialisation law: orthogonal Linear weights with gain 2 (MLP, d2d_ppo.py:71-72,89-90)
        or 3 (GRU head, :40), zero Linear biases, nn.GRU default U(-1/sqrt(H), 1/sqrt(H))."""
        for g in range(self.N):
            sd = {}
            if self.arch == L.NET_GRU:
                k = 1.0 / math.sqrt(self.H)
                for name in GRU_KEYS[:4]:
                    _, rows, cols = self._layout[g][GRU_KEYS.index(name)]
                    shape = (rows, cols) if cols > 1 or name.startswith("lstm.weight") else (rows,)
                    sd[name] = (torch.rand(*shape, generator=generator) * 2 - 1) * k
                sd["layers.0.weight"] = _orthogonal(self.H, self.H, 3, generator)
                sd["layers.0.bias"] = torch.zeros(self.H)
                last = "layers.2"
                if self.head_layers == 2:          # irdqn.py:66-72: same init law on every Linear
                    sd["layers.2.weight"] = _orthogonal(self.H, self.H, 3, generator)
                    sd["layers.2.bias"] = torch.zeros(self.H)
                    last = "layers.4"
                sd[last + ".weight"] = _orthogonal(self.O, self.H, 3, generator)
                sd[last + ".bias"] = torch.zeros(self.O)
            else:
                sd["linear1.weight"] = _orthogonal(self.H, self.in_dim[g], 2, generator)
                sd["linear1.bias"] = torch.zeros(self.H)
                sd["linear2.weight"] = _orthogonal(self.O, self.H, 2, generator)
                sd["linear2.bias"] = torch.zeros(self.O)
            self.load_state_dict(g, sd)

    def state_dict(self, agent):
        """Same keys and shapes as the reference module's state_dict (checkpoint compatible both ways)."""
        blk = self.params[agent].detach().cpu()
        out = {}
        for name, (off, rows, cols) in zip(self.keys, self._layout[agent]):
            t = blk[off:off + rows * cols].clone()
            out[name] = t.reshape(rows, cols) if name.endswith("weight") or "weight" in name else t
        return out

    def load_state_dict(self, agent, sd):
        blk = torch.zeros(self.stride, dtype=torch.float32)
        for name, (off, rows, cols) in zip(self.keys, self._layout[agent]):
            t = torch.as_tensor(sd[name], dtype=torch.float32).reshape(-1)
            if t.numel() != rows * cols:
                raise ValueError(f"{name}: expected {rows * cols} values, got {t.numel()}")
            blk[off:off + rows * cols] = t
        self.params[agent].copy_(blk.to(self.device))

    def training_state(self):
        """Parameters, Adam moments and step count as CPU copies (the ``agent_{i}.pth`` files hold the parameters
        only).  A handle that aliases another net set's buffers has nothing of its own: {}."""
        if self._owner is not None:
            return {}
        return {"params": self.params.cpu(), "adam_m": self.adam_m.cpu(), "adam_v": self.adam_v.cpu(),
                "adam_step": int(self.adam_step)}

    def load_training_state(self, d):
        """Inverse of ``training_state``: copies into the existing buffers, so handles that alias them see the
        restored values."""
        if self._owner is not None:
            if d:
                raise ValueError("this handle aliases another net set's parameters: load the owner")
            return
        for name in ("params", "adam_m", "adam_v"):
            t = d[name]
            if tuple(t.shape) != tuple(self.params.shape) or t.dtype != self.params.dtype:
                raise ValueError(f"{name}: expected {self.params.dtype} {tuple(self.params.shape)}, got "
                                 f"{t.dtype} {tuple(t.shape)}")
        for name in ("params", "adam_m", "adam_v"):
            getattr(self, name).copy_(d[name])
        self.adam_step = int(d["adam_step"])

    def tensor_view(self, buf, agent, name):
        off, rows, cols = self._layout[agent][self.keys.index(name)]
        v = buf[agent, off:off + rows * cols]
        return v.reshape(rows, cols) if "weight" in name else v

    # ---------------------------------------------------------------- kernels
    def forward(self, x, x_lead, t0, t1, padded, out=None, params=None):
        """Pre-activation outputs [t1 - t0, N, O, B] of time blocks [t0, t1) of the env-minor input matrix x.
        params: another [N, stride] parameter buffer of the same layout (a target network)."""
        if out is None:
            out = torch.empty((t1 - t0, self.N, self.O, self.B), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self._lib.d2d_net_forward(self._h, L.ptr(self.params if params is None else params), L.ptr(x),
                                              int(x_lead), int(t0), int(t1), int(padded), L.ptr(out),
                                              L.current_stream()))
        return out

    def rollout_step(self, x, x_lead, t, out=None):
        """Pre-activation outputs [1, N, O, B] of time block t (unpadded window), input projections cached across
        the steps of an episode.  Call with t = 0, 1, ... in order; parameters must stay fixed within the episode."""
        if out is None:
            out = torch.empty((1, self.N, self.O, self.B), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self._lib.d2d_net_rollout_step(self._h, L.ptr(self.params), L.ptr(x), int(x_lead), int(t),
                                                   L.ptr(out), L.current_stream()))
        return out

    def rollout_act(self, x, x_lead, t, dist_kind, act_mode, actions_t, logp_t, seed=0, env_offset=0, t_abs0=0,
                    logits_out=None):
        """select_action of all agents at time t in one call (d2d_net_rollout_act): forward on the unpadded window,
        then action (sampled / greedy / given) and log-prob into ``actions_t`` / ``logp_t`` ([N, B] blocks of time t).
        One kernel launch when the tensor-core window kernel takes the net."""
        with torch.cuda.device(self.device):
            L.check(self._lib.d2d_net_rollout_act(self._h, L.ptr(self.params), L.ptr(x), int(x_lead), int(t),
                                                  int(dist_kind), int(act_mode), L.ptr(actions_t), L.ptr(logp_t),
                                                  int(seed) & 0xFFFFFFFFFFFFFFFF, int(env_offset), int(t_abs0),
                                                  L.ptr(logits_out), L.current_stream()))

    def count_inexact_inputs(self, x, x_lead, t0, t1):
        """Device u64 scalar: inputs of time blocks [t0, t1) that are not exactly representable in bf16 (the guard of
        ``inputs_bf16_exact``, d2d_net_check_inputs)."""
        out = torch.zeros(1, dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self._lib.d2d_net_check_inputs(self._h, L.ptr(x), int(x_lead), int(t0), int(t1), L.ptr(out),
                                                   L.current_stream()))
        return out

    def zero_grad(self):
        self.grads.zero_()

    def policy_grad(self, x, x_lead, t0, t1, dist_kind, actions, logp_old, weight, weight_per_agent, cycle, inv_rows,
                    cliprange, beta, loss_sums, ratio_out=None):
        with torch.cuda.device(self.device):
            L.check(self._lib.d2d_ppo_policy_grad(
                self._h, L.ptr(self.params), L.ptr(x), int(x_lead), int(t0), int(t1), int(dist_kind), L.ptr(actions),
                L.ptr(logp_old), L.ptr(weight), int(weight_per_agent), L.ptr(cycle), float(inv_rows),
                float(cliprange), float(beta), L.ptr(self.grads), L.ptr(loss_sums), L.ptr(ratio_out),
                L.current_stream()))

    def value_grad(self, x, x_lead, t0, t1, padded, target, per_agent, inv_rows, loss_sum, value_out=None):
        with torch.cuda.device(self.device):
            L.check(self._lib.d2d_value_grad(
                self._h, L.ptr(self.params), L.ptr(x), int(x_lead), int(t0), int(t1), int(padded), L.ptr(target),
                int(per_agent), float(inv_rows), L.ptr(self.grads), L.ptr(loss_sum), L.ptr(value_out),
                L.current_stream()))

    def q_grad(self, x, x_lead, t0, t1, actions, target, loss_kind, inv_rows, loss_sum, q_out=None):
        """DQN.train_step up to the optimiser (d2d_q_grad): gradients of loss(Q[action], target) accumulated into
        ``grads``, the loss terms summed into ``loss_sum`` (f64 [N])."""
        with torch.cuda.device(self.device):
            L.check(self._lib.d2d_q_grad(self._h, L.ptr(self.params), L.ptr(x), int(x_lead), int(t0), int(t1),
                                         L.ptr(actions), L.ptr(target), int(loss_kind), float(inv_rows),
                                         L.ptr(self.grads), L.ptr(loss_sum), L.ptr(q_out), L.current_stream()))

    def adam(self, max_norm=0.0):
        """clip_grad_norm_(max_norm) per agent (if > 0) followed by one torch.optim.Adam step."""
        if self._owner is not None:
            raise RuntimeError("this handle aliases another net set's parameters: step the owner")
        self.adam_step += 1
        with torch.cuda.device(self.device):
            L.check(self._lib.d2d_adam_step_eps(L.ptr(self.params), L.ptr(self.adam_m), L.ptr(self.adam_v),
                                                L.ptr(self.grads), self.N, self.stride, self.lr, self.adam_eps,
                                                self.adam_step, float(max_norm), L.ptr(self._sqnorm),
                                                L.current_stream()))


def policy_head(logits, n_agents, n_envs, n_out, out_kind, dist_kind, act_mode, actions, logp, entropy=None,
                probs=None, seed=0, env_offset=0, t_abs0=0):
    """select_action / evaluate on pre-activation outputs [n_t, N, O, B] (csrc: policy_head_kernel)."""
    n_t = logits.shape[0]
    with torch.cuda.device(logits.device):
        L.check(L.lib().d2d_policy_head(n_agents, n_envs, n_out, n_t, out_kind, dist_kind, act_mode, L.ptr(logits),
                                        L.ptr(actions), L.ptr(logp), L.ptr(entropy), L.ptr(probs),
                                        int(seed) & 0xFFFFFFFFFFFFFFFF, int(env_offset), int(t_abs0),
                                        L.current_stream()))


def q_select(q, n_agents, n_envs, n_out, act_mode, epsilon, ready, n_random, action_idx, action_mask, seed=0,
             env_offset=0, t_abs=0):
    """DQN.act / DQN.predict for all agents and envs (d2d_q_select): Q-values [1, N, O, B] -> channel index u8 [N, B]
    and the one-hot channel bitmask the env kernels take."""
    mask_bytes = 0 if action_mask is None else action_mask.element_size()
    with torch.cuda.device(action_idx.device):
        L.check(L.lib().d2d_q_select(n_agents, n_envs, n_out, L.ptr(q), int(act_mode), float(epsilon), int(bool(ready)),
                                     int(n_random), L.ptr(action_idx), L.ptr(action_mask), mask_bytes,
                                     int(seed) & 0xFFFFFFFFFFFFFFFF, int(env_offset), int(t_abs), L.current_stream()))


def q_td_target(q_next, reward, done, gamma, out=None):
    """rewards + (1 - dones) * gamma * max_a Q_target(s') (irdqn.py:137-139): [1, N, O, B] -> f32 [N, B]."""
    _, N, O, B = q_next.shape
    if out is None:
        out = torch.empty((N, B), dtype=torch.float32, device=q_next.device)
    with torch.cuda.device(q_next.device):
        L.check(L.lib().d2d_q_td_target(N, B, O, L.ptr(q_next), L.ptr(reward), L.ptr(done), float(gamma), L.ptr(out),
                                        L.current_stream()))
    return out


def action_dtype(dist_kind, n_out):
    if dist_kind == L.DIST_CATEGORICAL or n_out <= 8:
        return torch.uint8
    return torch.int16 if n_out <= 16 else torch.int32


def returns_scan(reward, value, gamma, lam, last_shard, want_adv=True, want_ret=True):
    """compute_gae / discount_rewards scans -> (adv_raw f64 [T, n_cols, B] | None, ret_raw | None, stats [n_cols, 4])."""
    T, B = reward.shape
    n_cols = value.shape[1] if value is not None else 1
    dev = reward.device
    adv = torch.empty((T, n_cols, B), dtype=torch.float64, device=dev) if want_adv else None
    ret = torch.empty((T, n_cols, B), dtype=torch.float64, device=dev) if want_ret else None
    stats = torch.zeros((n_cols, 4), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        L.check(L.lib().d2d_returns_scan(L.ptr(reward), L.ptr(value), L.ptr(adv), L.ptr(ret), L.ptr(stats), T, B,
                                         n_cols, float(gamma), float(lam), int(last_shard), L.current_stream()))
    return adv, ret, stats


def returns_stats(reward, value, gamma, lam, last_shard, want_adv=True, want_ret=True):
    """Pass 1 of the two-pass scans: normalisation statistics only -> stats f64 [n_cols, 4]."""
    T, B = reward.shape
    n_cols = value.shape[1] if value is not None else 1
    stats = torch.zeros((n_cols, 4), dtype=torch.float64, device=reward.device)
    with torch.cuda.device(reward.device):
        L.check(L.lib().d2d_returns_stats(L.ptr(reward), L.ptr(value), L.ptr(stats), T, B, n_cols, float(gamma),
                                          float(lam), int(last_shard), int(want_adv), int(want_ret),
                                          L.current_stream()))
    return stats


def returns_norm_stats(stats, rows):
    """(adv (mean, std, flags), ret (mean, std, flags)) from the all-reduced [n_cols, 4] sums and the global row count
    (d2d_returns_norm_stats: one launch, everything stays on the device)."""
    n_cols, dev = stats.shape[0], stats.device
    f = torch.empty((4, n_cols), dtype=torch.float64, device=dev)
    flags = torch.empty((2, n_cols), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        L.check(L.lib().d2d_returns_norm_stats(L.ptr(stats), n_cols, float(rows), L.ptr(f[0]), L.ptr(f[1]),
                                               L.ptr(flags[0]), L.ptr(f[2]), L.ptr(f[3]), L.ptr(flags[1]),
                                               L.current_stream()))
    return (f[0], f[1], flags[0]), (f[2], f[3], flags[1])


def returns_emit(reward, value, gamma, lam, last_shard, adv_norm=None, ret_norm=None, adv_out=None, ret_out=None):
    """Pass 2: repeat the scans and write the normalised fp32 lambda-returns / returns [T, n_cols, B].
    adv_norm / ret_norm: (mean, std, flags) of ``PPOBase._norm_stats`` or None to skip that scan."""
    T, B = reward.shape
    n_cols = value.shape[1] if value is not None else 1
    dev = reward.device
    if adv_norm is not None and adv_out is None:
        adv_out = torch.empty((T, n_cols, B), dtype=torch.float32, device=dev)
    if ret_norm is not None and ret_out is None:
        ret_out = torch.empty((T, n_cols, B), dtype=torch.float32, device=dev)
    a = adv_norm if adv_norm is not None else (None, None, None)
    r = ret_norm if ret_norm is not None else (None, None, None)
    with torch.cuda.device(dev):
        L.check(L.lib().d2d_returns_emit(L.ptr(reward), L.ptr(value), L.ptr(adv_out if adv_norm is not None else None),
                                         L.ptr(ret_out if ret_norm is not None else None), L.ptr(a[0]), L.ptr(a[1]),
                                         L.ptr(a[2]), L.ptr(r[0]), L.ptr(r[1]), L.ptr(r[2]), T, B, n_cols,
                                         float(gamma), float(lam), int(last_shard), L.current_stream()))
    return adv_out, ret_out


def normalize(raw, mean, std, do_norm, fp32_math):
    T, n_cols, B = raw.shape
    out = torch.empty((T, n_cols, B), dtype=torch.float32, device=raw.device)
    with torch.cuda.device(raw.device):
        L.check(L.lib().d2d_normalize(L.ptr(raw), L.ptr(out), L.ptr(mean), L.ptr(std), L.ptr(do_norm), int(fp32_math),
                                      T, B, n_cols, L.current_stream()))
    return out
