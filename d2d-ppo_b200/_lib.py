"""ctypes binding of the C ABI in include/d2d_b200.h (libd2d_b200.so, built in-tree for sm_100a).

Loading fails loudly: there is no CPU or PyTorch fallback for any entry point.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libd2d_b200.so")

OK, ERR_INVALID, ERR_CUDA, ERR_STATE = 0, -1, -2, -3
ENV_COMBINATORIAL, ENV_SINGLE_CHANNEL, ENV_CHANNEL_SELECTION = 0, 1, 2
RNG_PHILOX, RNG_REPLAY = 0, 1
ARRIVAL_POISSON, ARRIVAL_BERNOULLI = 0, 1
MAX_AGENTS, MAX_CHANNELS, MAX_DEADLINE, POISSON_KMAX = 64, 32, 32, 16


class D2DError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libd2d_b200 error {code}: {msg}")
        self.code = code


class EnvConfig(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("n_envs", C.c_int32), ("n_agents", C.c_int32), ("n_channels", C.c_int32),
        ("episode_length", C.c_int32), ("homogeneous_size", C.c_int32), ("rng_mode", C.c_int32),
        ("reserved0", C.c_int32), ("seed", C.c_uint64), ("env_offset", C.c_uint64),
        ("deadlines", C.POINTER(C.c_int32)), ("arrival_kind", C.POINTER(C.c_int32)),
        ("arrival_active", C.POINTER(C.c_uint64)), ("poisson_cdf", C.POINTER(C.c_uint32)),
        ("bernoulli_thr", C.POINTER(C.c_uint64)), ("switch_thr", C.POINTER(C.c_uint32)),
        ("nbr_offset", C.POINTER(C.c_int32)), ("nbr_index", C.POINTER(C.c_int32)),
    ]


class NetConfig(C.Structure):
    _fields_ = [
        ("arch", C.c_int32), ("out_kind", C.c_int32), ("n_agents", C.c_int32), ("n_envs", C.c_int32),
        ("hidden", C.c_int32), ("n_out", C.c_int32), ("history_len", C.c_int32), ("in_rows", C.c_int32),
        ("in_dim", C.POINTER(C.c_int32)), ("in_off", C.POINTER(C.c_int32)), ("scratch_bytes", C.c_int64),
        ("inputs_bf16_exact", C.c_int32), ("head_layers", C.c_int32),
    ]


NET_MLP, NET_GRU = 0, 1
OUT_SOFTMAX, OUT_SIGMOID, OUT_IDENTITY = 0, 1, 2
DIST_BERNOULLI, DIST_CATEGORICAL = 0, 1
ACT_SAMPLE, ACT_GREEDY, ACT_GIVEN = 0, 1, 2
ACT_HOST_REFERENCE, ACT_HOST_DEVICE_LAYOUT = 0, 1
QLOSS_HUBER, QLOSS_MSE = 0, 1
SWITCH_ALL_TC, SWITCH_ENV_MULTISTEP, SWITCH_HOST_PACK = 5, 9, 10

_lib = None

_P = C.c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)
    "d2d_last_error": (C.c_char_p, []),
    "d2d_abi_version": (C.c_int, []),
    "d2d_launch_count": (C.c_uint64, []),
    "d2d_env_create": (C.c_int, [C.POINTER(EnvConfig), C.POINTER(_P)]),
    "d2d_env_destroy": (C.c_int, [_P]),
    "d2d_env_obs_rows": (C.c_int, [_P]),
    "d2d_env_obs_offset": (C.c_int, [_P, C.c_int]),
    "d2d_env_obs_dim": (C.c_int, [_P, C.c_int]),
    "d2d_env_state_rows": (C.c_int, [_P]),
    "d2d_env_timestep": (C.c_int, [_P]),
    "d2d_env_episode": (C.c_int64, [_P]),
    "d2d_env_set_episode": (C.c_int, [_P, C.c_int64]),
    "d2d_env_record_bytes": (C.c_int, [_P]),
    "d2d_env_mask_bytes": (C.c_int, [_P]),
    "d2d_env_set_replay": (C.c_int, [_P, _P, _P, C.c_int]),
    "d2d_env_reset": (C.c_int, [_P, _P, _P, _P]),
    "d2d_env_step": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "d2d_env_step_random_access": (C.c_int, [_P, C.c_double, _P, _P, _P, _P, _P, _P, _P]),
    "d2d_env_run_random_access": (C.c_int, [_P, C.c_double, C.c_int, C.c_int, _P, C.c_int64, _P, C.c_int64, _P, C.c_int64,
                                            C.c_int, _P, _P, C.POINTER(C.c_int)]),
    "d2d_env_step_host": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, _P, _P, C.POINTER(C.c_uint64)]),
    "d2d_env_host_wait": (C.c_int, [_P, C.c_uint64]),
    "d2d_env_host_pack_state": (C.c_int, [_P]),
    "d2d_pack_actions": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "d2d_set_host_threads": (C.c_int, [C.c_int]),
    "d2d_get_host_threads": (C.c_int, []),
    "d2d_pack_actions_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int]),
    "d2d_env_export_state": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "d2d_env_import_state": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "d2d_env_scores": (C.c_int, [_P, _P, _P, _P, _P]),
    "d2d_env_policy_edf": (C.c_int, [_P, C.c_int, _P, _P]),
    "d2d_net_create": (C.c_int, [C.POINTER(NetConfig), C.POINTER(_P)]),
    "d2d_net_destroy": (C.c_int, [_P]),
    "d2d_net_param_stride": (C.c_int64, [_P]),
    "d2d_net_num_tensors": (C.c_int, [_P]),
    "d2d_net_tensor": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int32),
                                 C.POINTER(C.c_int32)]),
    "d2d_net_forward": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "d2d_net_check_inputs": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "d2d_set_kernel_switch": (C.c_int, [C.c_int, C.c_int]),
    "d2d_get_kernel_switch": (C.c_int, [C.c_int]),
    "d2d_set_deterministic": (C.c_int, [C.c_int]),
    "d2d_get_deterministic": (C.c_int, []),
    "d2d_net_rollout_step": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, _P, _P]),
    "d2d_net_rollout_act": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_uint64, C.c_uint64,
                                      C.c_int, _P, _P]),
    "d2d_policy_head": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P,
                                  C.c_uint64, C.c_uint64, C.c_int, _P]),
    "d2d_ppo_policy_grad": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_int, _P,
                                      C.c_float, C.c_float, C.c_float, _P, _P, _P, _P]),
    "d2d_value_grad": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, C.c_float, _P, _P, _P,
                                 _P]),
    "d2d_adam_step": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int64, C.c_float, C.c_int, C.c_float, _P, _P]),
    "d2d_returns_scan": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int,
                                   _P]),
    "d2d_returns_stats": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int,
                                    C.c_int, _P]),
    "d2d_returns_norm_stats": (C.c_int, [_P, C.c_int, C.c_double, _P, _P, _P, _P, _P, _P, _P]),
    "d2d_returns_emit": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_double,
                                   C.c_double, C.c_int, _P]),
    "d2d_normalize": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "d2d_adam_step_eps": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int64, C.c_float, C.c_float, C.c_int, C.c_float, _P,
                                    _P]),
    "d2d_q_select": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, C.c_int, C.c_float, C.c_int, C.c_int, _P, _P, C.c_int,
                               C.c_uint64, C.c_uint64, C.c_int, _P]),
    "d2d_q_td_target": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_float, _P, _P]),
    "d2d_q_grad": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, C.c_float, _P, _P, _P, _P]),
    "d2d_replay_gather": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_int, _P, _P, _P, _P, _P, _P]),
}


def exported_symbols():
    """Names declared in include/d2d_b200.h that this binding expects (checked by the CPU tests)."""
    return sorted(_SIGNATURES)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the CUDA library has not been built. Run "
                "`python -c 'import __graft_entry__ as g; g.build()'` from the repo root. "
                "There is no CPU fallback for this path.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = res, args
        if handle.d2d_abi_version() != 1:
            raise ImportError("libd2d_b200.so ABI version mismatch; rebuild")
        # host thread pool of the host-buffer step: this rank's share of the CPUs it may run on (torchrun exports
        # LOCAL_WORLD_SIZE; the C library itself reads no environment variables)
        try:
            cpus = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
            share = max(1, cpus // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1"))))
            handle.d2d_set_host_threads(min(16, share))
        except (ValueError, OSError):
            pass
        _lib = handle
    return _lib


def check(code):
    if code != OK:
        raise D2DError(code, lib().d2d_last_error().decode("utf-8", "replace"))
    return code


def set_kernel_switch(which: int, enabled: bool) -> None:
    """A/B and debugging control of the SWITCH_* paths (d2d_set_kernel_switch); process-wide."""
    check(lib().d2d_set_kernel_switch(int(which), int(bool(enabled))))


def launch_count() -> int:
    return int(lib().d2d_launch_count())


def ptr(t):
    """Device (or host) address of a torch tensor, or NULL."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
