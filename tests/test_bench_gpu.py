"""bench.py --dump-outputs on the GPU: the saved outputs are those of the last timed step, as the numpy oracle computes
them from the bench's seeded inputs, so they are reproducible from run to run and --steps sets which step that is."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B = 4096


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                        "--warmup", "2", "--envs", str(B), "--no-configs", "--no-learner", "--no-cpu-baseline",
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert j["steps"] == steps
    return {f[:-4]: np.load(out_dir / f) for f in sorted(os.listdir(out_dir))}


def _oracle_steps(last_steps):
    """The bench's timed path on the numpy oracle: seed 42, a reset into episode 0, then LEAD_IN + K fused
    random-access steps; outputs after step LEAD_IN + K for every K in last_steps."""
    import bench
    from d2d_ppo_b200 import presets
    from oracle import philox_np as px
    from oracle.envs_np import CombinatorialOracle, PhiloxSource
    kw = presets.combinatorial_kwargs("setup_8_channels", load=bench.LOAD)
    assert bench.LEAD_IN + max(last_steps) < kw["episode_length"]         # no auto reset inside the run
    orc = CombinatorialOracle(n_envs=B, source=PhiloxSource(B, 42), **kw)
    orc.reset()
    envs, thr, out = np.arange(B), px.thr16(bench.TP), {}
    for t in range(1, bench.LEAD_IN + max(last_steps) + 1):
        a = np.stack([px.lanes16(42, envs, t, k, px.PURPOSE_POLICY, bench.N_CHANNELS) < thr
                      for k in range(bench.N_AGENTS)], axis=1)
        obs, _, rew, _, _ = orc.step(a)
        if t - bench.LEAD_IN in last_steps:
            out[t - bench.LEAD_IN] = {"obs": np.concatenate(obs, axis=1).T, "reward": rew[:, 0],
                                      "discarded": orc.discarded.copy(), "received": orc.received.copy()}
    return out


def test_dump_outputs_are_the_last_timed_step(tmp_path, cuda_device):
    dumps = {k: _bench(tmp_path / f"steps{k}", k) for k in (7, 8)}
    ref = _oracle_steps(tuple(dumps))
    for k, d in dumps.items():
        assert set(d) == {"env_index", "obs", "reward", "discarded", "received"}
        assert sum(x.nbytes for x in d.values()) <= 64 << 20
        assert all(x.dtype in (np.float32, np.float64) for x in d.values())
        assert np.array_equal(d["env_index"], np.arange(B))               # fewer envs than the sample: all of them
        for name, want in ref[k].items():
            assert np.array_equal(d[name], want.astype(np.float32)), (k, name)
        assert d["received"].sum() > 0
    assert not np.array_equal(dumps[7]["obs"], dumps[8]["obs"])
