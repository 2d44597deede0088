"""Training-state files without a GPU: the commit order of a checkpoint, config checks, and the replay ring's state
(the agents' resume runs are in test_resume_gpu.py)."""
import os

import numpy as np
import pytest
import torch

CFG = {"class": "iPPO", "n_agents": 3, "hidden_size": 64, "history_len": 4, "n_envs": 8, "episode_length": 5,
       "obs_layout": [12, [0, 4, 8], [4, 4, 4]], "seed": 1, "world_size": 1}


def _save(path, value):
    from d2d_ppo_b200.algorithms import _ckpt
    _ckpt.save(str(path), CFG, {"x": torch.full((4,), float(value)), "n": value}, {"local": [value]}, "cpu")


def test_checkpoint_round_trip_and_weights_only(tmp_path):
    from d2d_ppo_b200.algorithms import _ckpt
    _save(tmp_path, 1)
    _save(tmp_path, 2)
    files = sorted(os.listdir(tmp_path))
    assert len(files) == 2 and _ckpt.MAIN_FILE in files          # the older rank file is gone
    for f in files:
        torch.load(tmp_path / f, weights_only=True)
    rep, loc = _ckpt.load(str(tmp_path), CFG)
    assert rep["n"] == 2 and torch.equal(rep["x"], torch.full((4,), 2.0)) and loc == {"local": [2]}


@pytest.mark.parametrize("field,value", [("hidden_size", 32), ("n_envs", 16), ("class", "D2DPPO"), ("world_size", 2)])
def test_checkpoint_rejects_other_settings(tmp_path, field, value):
    from d2d_ppo_b200.algorithms import _ckpt
    _save(tmp_path, 1)
    with pytest.raises(ValueError, match=field):
        _ckpt.load(str(tmp_path), dict(CFG, **{field: value}))


@pytest.mark.parametrize("fail_at", [1, 2])
def test_interrupted_write_keeps_previous_checkpoint(tmp_path, monkeypatch, fail_at):
    """A write that dies part way (first the rank file, then rank 0's file) leaves the previous checkpoint whole."""
    from d2d_ppo_b200.algorithms import _ckpt
    _save(tmp_path, 1)
    real, calls = torch.save, []

    def flaky(obj, f):
        calls.append(f)
        if len(calls) == fail_at:
            with open(f, "wb") as fh:
                fh.write(b"partial")
            raise OSError("disk full")
        real(obj, f)
    monkeypatch.setattr(torch, "save", flaky)
    with pytest.raises(OSError):
        _save(tmp_path, 2)
    monkeypatch.setattr(torch, "save", real)
    rep, loc = _ckpt.load(str(tmp_path), CFG)
    assert rep["n"] == 1 and loc == {"local": [1]}
    assert not [f for f in os.listdir(tmp_path) if ".tmp" in f]


def test_replay_state_round_trip(tmp_path):
    """Only the filled slots are stored, in ring order; a restored ring holds them in the same slots and its sampling
    generator continues the same stream."""
    from d2d_ppo_b200.algorithms.irdqn import ReplayBuffer
    kw = dict(n_envs=3, n_agents=2, episode_length=4, obs_rows=5, seed=9)
    a = ReplayBuffer(3 * 4 * 4, "cpu", **kw)                         # 4 slots
    g = torch.Generator().manual_seed(0)
    for k in range(6):                                               # wraps: head 2, slots 2, 3, 0, 1 in ring order
        a.add_episode(torch.randn((5, 5, 3), generator=g), torch.randint(0, 8, (4, 2, 3), generator=g).byte(),
                      torch.randint(-1, 2, (4, 3), generator=g).int())
        if k == 1:
            partial = a.state_dict()
            assert partial["obs"].shape[0] == 2
    a._rng.integers(0, 10, 7)
    d = a.state_dict()
    assert d["obs"].shape[0] == 4 and d["head"] == 2
    assert torch.equal(d["obs"][0], a.obs[2]) and torch.equal(d["rew"][3], a.rew[1])
    torch.save(d, tmp_path / "replay.pt")
    d = torch.load(tmp_path / "replay.pt", weights_only=True)
    b = ReplayBuffer(3 * 4 * 4, "cpu", **kw)
    b.load_state_dict(d)
    assert (b.head, b.n_stored) == (a.head, a.n_stored)
    for k in ("obs", "act", "rew"):
        assert torch.equal(getattr(a, k), getattr(b, k))
    assert np.array_equal(a._rng.integers(0, 1000, 50), b._rng.integers(0, 1000, 50))
    c = ReplayBuffer(3 * 4 * 4, "cpu", **kw)
    c.load_state_dict(partial)
    assert (c.head, c.n_stored) == (2, 2)
    with pytest.raises(ValueError, match="n_slots"):
        ReplayBuffer(3 * 4 * 8, "cpu", **kw).load_state_dict(d)


def test_float_lists_round_trip_exactly_and_convert_only_new_values():
    from d2d_ppo_b200.algorithms._ckpt import FloatLists
    f = FloatLists()
    scores = [0.1, float("nan"), 1 / 3]
    t = f.to_tensor("s", scores)
    assert t.dtype == torch.float64 and t.shape == (3,)
    scores += [2 / 7]
    t2 = f.to_tensor("s", scores)
    assert torch.equal(t2[:3].nan_to_num(), t.nan_to_num()) and t2[3].item() == 2 / 7
    assert f.to_tensor("s", scores) is t2                       # nothing new: no conversion
    losses = [[0.5, -1.25], [1e-300, 3.0]]                        # D2DPPO: one [N] row per epoch
    back = FloatLists().to_list("l", f.to_tensor("l", losses))
    assert back == losses
    back = FloatLists().to_list("s", t2)
    assert np.array_equal(back, scores, equal_nan=True) and all(type(v) is float for v in back)
    assert f.to_tensor("s", list(scores)).shape == (4,)         # another list object: converted afresh
    assert FloatLists().to_tensor("e", []).shape == (0,)
