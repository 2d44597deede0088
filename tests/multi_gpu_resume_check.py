"""Run under torchrun on >= 2 GPUs: a sharded run that is checkpointed, dropped and resumed from its training state
(rank 0's replicated file plus one rank-local file per rank) continues like the uninterrupted sharded run.  The
counters and list lengths match exactly; parameters and losses agree within the tolerances of multi_gpu_check.py
(sharded runs make no bit-exact promise).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 \
        tests/multi_gpu_resume_check.py
"""
import os
import shutil
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import d2d_ppo_b200  # noqa: E402
from d2d_ppo_b200 import presets  # noqa: E402
from d2d_ppo_b200.algorithms.d2d_ppo import D2DPPO  # noqa: E402
from d2d_ppo_b200.algorithms.irdqn import iRDQN  # noqa: E402
from d2d_ppo_b200.envs import CombinatorialEnv  # noqa: E402


def make_d2dppo(Bw, offset, dev):
    kw = presets.combinatorial_kwargs("setup_8_channels", load=0.5, episode_length=30)
    env = CombinatorialEnv(n_envs=Bw, device=dev, seed=21, env_offset=offset, **kw)
    np.random.seed(5)
    return D2DPPO(env, hidden_size=32, gamma=0.6, policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=True,
                  history_len=4, early_stopping=False, seed=5)


def train_d2dppo(ag, n, **kw):
    return ag.train(num_iter=n, num_episodes=ag.B, n_epoch=2, test_freq=2, **kw)


def make_irdqn(Bw, offset, dev):
    kw = presets.combinatorial_kwargs("setup_8_channels", load=0.5, episode_length=20)
    env = CombinatorialEnv(n_envs=Bw, device=dev, seed=23, env_offset=offset, **kw)
    return iRDQN(env, history_len=4, replay_start_size=1, replay_buffer_size=Bw * 20 * 4, gamma=0.6,
                 update_target_frequency=2, minibatch_size=16, learning_rate=1e-3, loss="huber", early_stopping=False,
                 hidden_size=32, seed=6)


def train_irdqn(ag, n, **kw):
    return ag.train(n, early_stopping=False, **kw)


def close(a, b, what):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert np.allclose(a, b, rtol=1e-4, atol=1e-6), (what, a, b)


def check(name, make, run, n_total, n_cut, rank, world, dev, ck):
    Bw = 256 // world
    full = make(Bw, rank * Bw, dev)
    want = run(full, n_total)
    cut = make(Bw, rank * Bw, dev)
    run(cut, n_cut, checkpoint_path=ck, checkpoint_freq=1)
    del cut
    resumed = make(Bw, rank * Bw, dev)
    np.random.seed(1000 + rank)               # the stored np.random state must win
    got = run(resumed, n_total, checkpoint_path=ck, resume=True)
    torch.cuda.synchronize()
    assert [len(x) for x in got] == [len(x) for x in want], name
    assert resumed.env.episode == full.env.episode, name
    pos = "next_episode" if name == "irdqn" else "next_iter"
    assert resumed._progress[pos] == full._progress[pos] == n_total, name
    if name == "irdqn":
        assert (resumed._episode, resumed.epsilon) == (full._episode, full.epsilon)
        rb, fb = resumed.replay_buffer, full.replay_buffer
        assert (rb.head, rb.n_stored) == (fb.head, fb.n_stored) and len(resumed.losses) == len(full.losses)
        close(torch.stack(resumed.losses).cpu(), torch.stack(full.losses).cpu(), "losses")
        pairs = [(resumed.network.params, full.network.params), (resumed.target_params, full.target_params)]
    else:
        assert resumed._iter == full._iter
        close(got[2], want[2], "policy losses")
        close(got[3], want[3], "value losses")
        pairs = [(resumed.policies.params, full.policies.params), (resumed.critic.params, full.critic.params)]
    d = max((a - b).abs().max().item() for a, b in pairs)
    assert d < 5e-5, (name, d)
    close(got[0], want[0], "episode scores")              # rank-local: this rank's envs only
    dist.barrier()                            # every rank has removed its superseded rank file
    files = sorted(f for f in os.listdir(ck) if f.startswith("training_state"))
    assert len(files) == 1 + world, files     # rank 0's file and one rank-local file per rank
    if rank == 0:
        print(f"{name}: {world} ranks x {Bw} envs, cut after {n_cut} of {n_total} and resumed == uninterrupted "
              f"(counters and lengths equal, max |param diff| {d:.2e})")
    dist.barrier()


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    d2d_ppo_b200.use_deterministic_algorithms(True)
    holder = [tempfile.mkdtemp(prefix="resume_check_") if rank == 0 else None]
    dist.broadcast_object_list(holder, src=0)
    root = holder[0]
    try:
        check("d2dppo", make_d2dppo, train_d2dppo, 4, 2, rank, world, dev, os.path.join(root, "d2dppo"))
        check("irdqn", make_irdqn, train_irdqn, 6, 3, rank, world, dev, os.path.join(root, "irdqn"))
    finally:
        dist.barrier()
        if rank == 0:
            shutil.rmtree(root, ignore_errors=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
