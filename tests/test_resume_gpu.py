"""Save and resume the full training state: in deterministic mode a run cut after two iterations and continued in a
fresh process equals the uninterrupted run bit for bit; in default mode save -> load restores every tensor and counter
exactly; stored runs that stopped early return at once; files of another setup are rejected."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from test_deterministic_gpu import _c3_env, _sel_env

pytestmark = pytest.mark.gpu
TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
CASES = ["ippo_c3", "d2dppo_c3", "ippo_sel", "irdqn_c3"]


@pytest.fixture
def deterministic():
    import d2d_ppo_b200
    before = d2d_ppo_b200.are_deterministic_algorithms_enabled()
    d2d_ppo_b200.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        d2d_ppo_b200.use_deterministic_algorithms(before)


def build(case, dev, save_path=None, hidden=64, B=256, cls=None):
    """The agent of a case with small shapes (tests/test_deterministic_gpu.py); np.random seeded as the reference
    scripts do."""
    from d2d_ppo_b200.algorithms.d2d_ppo import D2DPPO
    from d2d_ppo_b200.algorithms.ippo import iPPO
    from d2d_ppo_b200.algorithms.irdqn import iRDQN
    np.random.seed(5)
    if case == "irdqn_c3":
        # replay_start_size 0, target sync every 2nd episode: optimiser steps at episodes 0, 1 | 2, 3 and target syncs
        # at 0 | 2 on both sides of a cut after episode 2
        return iRDQN(_c3_env(dev, 64, 20, seed=2), history_len=3, replay_start_size=0, replay_buffer_size=10 ** 5,
                     gamma=0.5, update_target_frequency=2, minibatch_size=32, learning_rate=1e-3,
                     early_stopping=False, hidden_size=hidden, seed=4)
    env = (_sel_env if case == "ippo_sel" else _c3_env)(dev, B, 20)
    kw = dict(hidden_size=hidden, gamma=0.6, policy_lr=3e-4, value_lr=1e-3, useRNN=True,
              combinatorial=env.action_kind == "bernoulli_mask", history_len=6, early_stopping=False,
              save_path=save_path, seed=7)
    cls = cls or (D2DPPO if case.startswith("d2dppo") else iPPO)
    return cls(env, beta_entropy=0.01, **kw) if cls is D2DPPO else cls(env, **kw)


def train(ag, n, **kw):
    from d2d_ppo_b200.algorithms.d2d_ppo import D2DPPO
    from d2d_ppo_b200.algorithms.irdqn import iRDQN
    if isinstance(ag, iRDQN):
        return ag.train(n, early_stopping=False, **kw)
    if isinstance(ag, D2DPPO):
        return ag.train(num_iter=n, num_episodes=ag.B, n_epoch=2, test_freq=1, **kw)
    return ag.train(num_iter=n, n_epoch=2, num_episodes=ag.B, test_freq=1, **kw)


def snapshot(ag, res=None):
    """Every tensor and counter the training state covers, as CPU copies, then a following test()."""
    from d2d_ppo_b200.algorithms.irdqn import iRDQN
    torch.cuda.synchronize()
    out = {"res": res, "env_episode": ag.env.episode}
    if isinstance(ag, iRDQN):
        out.update(net=ag.network.training_state(), target=ag.target_params.cpu(), epsilon=ag.epsilon,
                   episode=ag._episode, losses=[t.cpu() for t in ag.losses], replay=ag.replay_buffer.state_dict())
    else:
        out.update(nets={k: getattr(ag, k).training_state() for k in ag._NET_SETS}, iter=ag._iter)
        if hasattr(ag, "_np_rng"):            # D2DPPO's HAPPO order comes from the global np.random
            out["np_random"] = np.random.get_state(legacy=False)["state"]["key"].tolist()
    out["test"] = ag.test(50)
    return out


def assert_same(a, b, where="state"):
    if isinstance(a, dict):
        assert a.keys() == b.keys(), where
        for k in a:
            assert_same(a[k], b[k], f"{where}.{k}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), where
        for i, (x, y) in enumerate(zip(a, b)):
            assert_same(x, y, f"{where}[{i}]")
    elif torch.is_tensor(a):
        assert torch.equal(a, b), where
    elif isinstance(a, float):
        assert np.array_equal(a, b, equal_nan=True), (where, a, b)
    else:
        assert a == b, (where, a, b)


_CHILD = """
import sys, numpy as np, torch
sys.path[:0] = [{tests!r}, {root!r}]
import d2d_ppo_b200
from test_resume_gpu import build, snapshot, train
d2d_ppo_b200.use_deterministic_algorithms(True)
ag = build({case!r}, torch.device("cuda", 0), save_path={ck!r})
np.random.seed(12345)                     # the stored run's np.random state must win
res = train(ag, 4, checkpoint_path={ck!r}, checkpoint_freq=1, resume=True)
torch.save(snapshot(ag, res), {out!r})
"""


@pytest.mark.parametrize("case", CASES)
def test_resume_in_fresh_process_is_bit_identical(case, deterministic, tmp_path, cuda_device):
    full = build(case, cuda_device, save_path=str(tmp_path / "full"))
    want = snapshot(full, train(full, 4))
    ck = str(tmp_path / "ck")
    first = build(case, cuda_device, save_path=ck)
    res2 = train(first, 2, checkpoint_path=ck, checkpoint_freq=1)
    assert len(res2[0]) == 2 * first.B
    del first
    out = str(tmp_path / "resumed.pt")
    r = subprocess.run([sys.executable, "-c", _CHILD.format(tests=TESTS, root=ROOT, case=case, ck=ck, out=out)],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    got = torch.load(out, weights_only=False)
    assert_same(got, want)
    for f in os.listdir(ck):                  # the training-state files load without unpickling code
        if f.startswith("training_state"):
            torch.load(os.path.join(ck, f), map_location="cpu", weights_only=True)


@pytest.mark.parametrize("case", ["d2dppo_c3", "irdqn_c3"])
def test_default_mode_save_load_restores_state_exactly(case, tmp_path, cuda_device):
    import d2d_ppo_b200
    assert not d2d_ppo_b200.are_deterministic_algorithms_enabled()
    a = build(case, cuda_device)
    train(a, 2)
    a.save_training_state(str(tmp_path))
    want = snapshot(a)
    b = build(case, cuda_device)
    np.random.seed(999)
    b.load_training_state(str(tmp_path))
    got = snapshot(b)
    want.pop("test"), got.pop("test")          # default-mode continuations differ in the last bits, as two runs do
    assert_same(got, want)
    assert_same(b._progress, a._progress)


@pytest.mark.parametrize("case", ["ippo_c3", "irdqn_c3"])
def test_resume_after_early_stop_returns_at_once(case, tmp_path, cuda_device):
    from d2d_ppo_b200 import _lib as L
    a = build(case, cuda_device)
    a.early_stopping = True
    real = a.test
    a.test = lambda n: (1.0,) + tuple(real(n)[1:])       # a perfect test score fires early stopping
    kw = dict(checkpoint_path=str(tmp_path), checkpoint_freq=10, resume=True)
    res = train(a, 4, **kw) if case != "irdqn_c3" else a.train(4, early_stopping=True, **kw)
    assert a._progress["stopped"]
    b = build(case, cuda_device)
    n0 = L.launch_count()
    res_b = train(b, 4, **kw) if case != "irdqn_c3" else b.train(4, early_stopping=True, **kw)
    assert L.launch_count() == n0              # nothing ran
    assert_same(list(res_b), list(res))
    assert b.env.episode == a.env.episode


@pytest.mark.parametrize("field", ["hidden_size", "n_envs", "class"])
def test_load_rejects_other_setup(field, tmp_path, cuda_device):
    from d2d_ppo_b200.algorithms.d2d_ppo import D2DPPO
    a = build("ippo_c3", cuda_device, B=64)
    train(a, 1)
    a.save_training_state(str(tmp_path))
    kw = {"hidden_size": dict(hidden=32, B=64), "n_envs": dict(B=32), "class": dict(B=64, cls=D2DPPO)}[field]
    b = build("ippo_c3", cuda_device, **kw)
    with pytest.raises(ValueError, match=field):
        b.load_training_state(str(tmp_path))


def test_failed_write_keeps_previous_checkpoint(tmp_path, monkeypatch, cuda_device):
    a = build("irdqn_c3", cuda_device)
    train(a, 2, checkpoint_path=str(tmp_path), checkpoint_freq=1)
    want = snapshot(a)
    want.pop("test")
    train(a, 3, checkpoint_path=str(tmp_path), resume=True)     # one more episode, not checkpointed
    real = torch.save

    def dies_part_way(obj, f):
        with open(f, "wb") as fh:
            fh.write(b"\x80partial")
        raise OSError("killed")
    for n_ok in (0, 1):                        # dies in the rank file, then in rank 0's file
        calls = []

        def save(obj, f):
            calls.append(f)
            return real(obj, f) if len(calls) <= n_ok else dies_part_way(obj, f)
        monkeypatch.setattr(torch, "save", save)
        with pytest.raises(OSError):
            a.save_training_state(str(tmp_path))
        monkeypatch.setattr(torch, "save", real)
        b = build("irdqn_c3", cuda_device)
        b.load_training_state(str(tmp_path))
        got = snapshot(b)
        got.pop("test")
        assert_same(got, want)


@pytest.mark.parametrize("learner", ["d2dppo", "irdqn"])
def test_driver_rerun_with_resume_repeats_only_the_evaluation(learner, deterministic, tmp_path, cuda_device):
    """xp_load(resume=True) run twice: the second call finds every load finished, returns the stored training lists
    and repeats the final reload + test() on the same env episodes."""
    from d2d_ppo_b200 import experiments as X
    kw = dict(out_dir=str(tmp_path), learner=learner, loads=[0.5], num_iter=3, n_epoch=1, n_envs=8, test_freq=2,
              test_episodes=8, device=cuda_device, resume=True)
    np.random.seed(0)
    first = X.xp_load(**kw)
    folder = os.path.join(str(tmp_path), "models_mcappo8_seed_0_load_0.5")
    assert "training_state.pt" in os.listdir(folder)
    np.random.seed(1)
    again = X.xp_load(**kw)
    assert_same(again["training"], first["training"])
    for k in ("scores", "jains"):
        assert np.array_equal(again[k], first[k])


@pytest.mark.parametrize("case", ["ippo_c3", "irdqn_c3"])
def test_checkpoints_follow_iterations_0_k_2k_and_the_last(case, tmp_path, cuda_device, monkeypatch):
    """With checkpoint_freq = k = test_freq a checkpoint follows each test iteration, whose best-model files then
    belong to the stored run."""
    a = build(case, cuda_device, B=64)
    pos = "next_episode" if case == "irdqn_c3" else "next_iter"
    seen = []
    monkeypatch.setattr(a, "save_training_state", lambda path: seen.append(a._progress[pos]))
    train(a, 6, checkpoint_path=str(tmp_path), checkpoint_freq=4)
    assert seen == [1, 5, 6]
