"""Training-state files of the learners: everything that decides how a seeded run continues, so that an interrupted
run resumes where its last checkpoint left it.

A checkpoint directory holds one file of replicated state, written by rank 0 (``training_state.pt``), and one file of
rank-local state per rank (``training_state.rank{r}.{tag}.pt``: the rank's own episode scores and, for iRDQN, its
replay shard).  Every file is written to a temporary name, flushed to disk (fsync) and moved into place with
``os.replace``.  The rank files are written first; rank 0's file names their ``tag`` and is replaced last, so it is the
commit point: a job killed at any moment, or a node that crashes, leaves the previous checkpoint complete and loadable.
Rank files of older tags are removed only after the commit.  A rank whose write fails makes every rank raise instead
of waiting for it.  The files hold tensors, ints, floats, strings, lists and dicts only and load with
``torch.load(..., weights_only=True)``; the long float lists (episode scores, losses) are stored as float64 tensors.
"""
from __future__ import annotations

import glob
import os

import numpy as np
import torch

from . import _dist

FORMAT_VERSION = 1
MAIN_FILE = "training_state.pt"


def _rank_file(path, rank, tag):
    return os.path.join(path, f"training_state.rank{rank}.{tag}.pt")


def config(agent):
    """The settings a stored training state must match: they fix the shapes of the state, or (seed, world size) the
    streams a continuation draws.  n_envs is per rank."""
    return {"class": type(agent).__name__, "n_agents": agent.n_agents, "hidden_size": agent.hidden_size,
            "history_len": agent.history_len, "n_envs": agent.B, "episode_length": agent.T,
            "obs_layout": [agent.obs_rows, list(agent.obs_off), list(agent.obs_dim)], "seed": agent.seed,
            "world_size": _dist.world_size()}


def exists(path):
    return path is not None and os.path.exists(os.path.join(path, MAIN_FILE))


def _fsync(path):
    fd = os.open(path, os.O_RDONLY)
    try:
        os.fsync(fd)
    finally:
        os.close(fd)


def atomic_save(obj, file):
    """torch.save to a temporary name in the same directory, fsync, then os.replace and fsync of the directory:
    ``file`` is either its old content or the complete new one, also after a crash of the node."""
    tmp = f"{file}.tmp.{os.getpid()}"
    try:
        torch.save(obj, tmp)
        _fsync(tmp)
        os.replace(tmp, file)
    except BaseException:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise
    _fsync(os.path.dirname(file) or ".")


def _on_every_rank(write, device):
    """Run ``write``; then every rank learns whether some rank failed, and all of them raise if one did (a rank whose
    write failed raises its own error).  The count's all-reduce is also the barrier between the two phases of a save."""
    err = None
    try:
        write()
    except Exception as e:          # noqa: BLE001 -- re-raised below, after the other ranks were told
        err = e
    failed = int(_dist.all_reduce_sum_(torch.tensor([int(err is not None)], dtype=torch.int32, device=device)).item())
    if err is not None:
        raise err
    if failed:
        raise RuntimeError(f"training state not saved: the write failed on {failed} other rank(s)")


def save(path, config, replicated, local, device):
    """Write one checkpoint.  config: the settings ``load`` checks (``config``); replicated: rank 0's state; local:
    this rank's state.  Collective when a process group is active."""
    rank = _dist.rank()
    os.makedirs(path, exist_ok=True)
    tag = f"{_dist.broadcast_token(device):012x}"

    def commit():
        if rank == 0:
            atomic_save({"format": FORMAT_VERSION, "config": config, "tag": tag, "state": replicated},
                        os.path.join(path, MAIN_FILE))
    _on_every_rank(lambda: atomic_save({"format": FORMAT_VERSION, "config": config, "state": local},
                                       _rank_file(path, rank, tag)), device)
    _on_every_rank(commit, device)
    for old in glob.glob(_rank_file(path, rank, "*")):
        if old != _rank_file(path, rank, tag):
            os.remove(old)


def _check(file, d, config):
    if not isinstance(d, dict) or d.get("format") != FORMAT_VERSION:
        raise ValueError(f"{file}: format {d.get('format') if isinstance(d, dict) else None!r} is not the training-"
                         f"state format {FORMAT_VERSION}")
    stored = d["config"]
    for key, want in config.items():
        if stored.get(key) != want:
            raise ValueError(f"{file}: {key} is {stored.get(key)!r} in the training state but {want!r} here")


def load(path, config):
    """(replicated, local) state of the checkpoint in ``path``; ValueError names the first setting that differs."""
    main = os.path.join(path, MAIN_FILE)
    d = torch.load(main, map_location="cpu", weights_only=True)
    _check(main, d, {k: v for k, v in config.items() if k != "n_envs"})
    file = _rank_file(path, _dist.rank(), d["tag"])
    r = torch.load(file, map_location="cpu", weights_only=True)
    _check(file, r, config)
    return d["state"], r["state"]


class FloatLists:
    """The append-only float lists a checkpoint stores (episode scores, test scores, losses) as float64 tensors, which
    round-trip exactly, pickle in bulk and load fast with ``weights_only=True`` (a list of floats pickles and unpickles
    value by value).  A run's lists only grow between saves, so each save converts only the values appended since the
    previous one."""

    def __init__(self):
        self._seen = {}             # key -> (the list object, its values so far as a tensor)

    def to_tensor(self, key, values):
        lst, t = self._seen.get(key, (None, None))
        if lst is not values or t.shape[0] > len(values):
            t = None
        n = 0 if t is None else t.shape[0]
        if t is None or n < len(values):
            new = torch.from_numpy(np.asarray(values[n:], dtype=np.float64))
            t = new if not n else torch.cat([t, new])
        self._seen[key] = (values, t)
        return t

    def to_list(self, key, t):
        values = t.tolist()
        self._seen[key] = (values, t)
        return values


def plain(x):
    """numpy RNG states (bit_generator.state, np.random.get_state(legacy=False)) with their arrays as lists."""
    if isinstance(x, dict):
        return {k: plain(v) for k, v in x.items()}
    if isinstance(x, np.ndarray):
        return x.tolist()
    if isinstance(x, np.generic):
        return x.item()
    return x
