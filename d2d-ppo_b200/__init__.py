"""d2d-ppo_b200: B200-native hot path of benrobaglia/D2D-PPO.

Lockstep step/reset of the device-to-device channel-access environments and the PPO / IPPO
rollout-and-update loop, as hand-written sm_100a CUDA kernels behind a C ABI
(``include/d2d_b200.h`` -> ``libd2d_b200.so``), with the reference's Python env / agent API on top.

There is no CPU fallback: importing the env or agent classes loads the CUDA library and raises if it
has not been built (``python __graft_entry__.py`` / ``d2d_ppo_b200._build.build()``).
"""
__version__ = "0.1.0"

from . import spaces  # noqa: F401


def use_deterministic_algorithms(mode: bool) -> None:
    """Turn the learner's deterministic mode on or off (process-wide, off by default; may change between calls).

    With it on, every floating-point sum of the learner runs in a fixed order instead of through atomics, so a seeded
    single-GPU run gives bit-identical parameters, Adam moments, losses, scores and test() results with the same build,
    GPU model, seeds, n_envs and scratch_bytes.  D2DPPO draws its HAPPO agent order from the global np.random: seed it
    too.  The cost is L x the d(gi) scratch, one more pass over it per chunk and a few tiny launches
    (include/d2d_b200.h, d2d_set_deterministic).
    """
    from . import _lib
    _lib.check(_lib.lib().d2d_set_deterministic(int(bool(mode))))


def are_deterministic_algorithms_enabled() -> bool:
    """Whether the learner's deterministic mode is on (see use_deterministic_algorithms)."""
    from . import _lib
    return bool(_lib.lib().d2d_get_deterministic())
