"""The reference's experiment drivers as functions (SURVEY.md section 8f, row 2).

Each function reproduces one script of the reference -- same environment construction, learner hyper-parameters,
sweep, evaluation calls and result-dict layout (pickled to the same relative path) -- on the batched CUDA path:

* ``xp_load``            <- xp_load.py:31-161          D2DPPO (or iPPO) over ``loads_list`` on the 8-channel env
* ``xp_n_agents``        <- xp_n_agents.py:35-170      N-agent sweep (C = 4, deadlines 7) with the random-access
                                                        baseline, or D2DPPO / iPPO (the commented-out blocks)
* ``run_ma_baselines``   <- run_ma_baselines.py:21-97  setup.p written, CombinatorialRandomAccess over ``loads_list``
* ``xp_gamma``           <- xp_gamma.py:30-106         iPPO discount-factor sweep on ChannelSelectionEnv
* ``run_ippo_combinatorial`` <- run_ippo_combinatorial.py:65-94  iPPO on the 16-channel env

``n_envs`` plays the role of the reference's ``num_episodes`` (one lockstep env per episode of a rollout); the
defaults are the reference's values so that a run is comparable with its published curves, and every size can be
scaled down for a smoke run (``num_iter``, ``test_episodes``, ...).  Seeds: the reference fixes ``random`` and
``np.random`` to 42 (xp_load.py:12-14); here the env and learner Philox / init seeds derive from ``seed``.

    python -m d2d_ppo_b200.experiments xp_load --num-iter 20 --n-envs 64 --out results/
"""
from __future__ import annotations

import os
import pickle

import numpy as np

from . import presets


def _mk(path):
    os.makedirs(path, exist_ok=True)
    return path


def _learner(kind, env, save_path, seed, **kw):
    from .algorithms.d2d_ppo import D2DPPO
    from .algorithms.ippo import iPPO
    cls = {"d2dppo": D2DPPO, "ippo": iPPO}[kind]
    return cls(env, save_path=save_path, seed=seed, **kw)


def _ckpt_kw(resume, folder, freq):
    """train() arguments of a resumable run: the training state goes to the run's model folder after every
    ``freq``-th iteration, i.e. right after each test iteration when freq = test_freq (and after the last one), and a
    rerun continues from it; a run that had finished returns its stored lists at once, so only the evaluation after it
    repeats."""
    return dict(checkpoint_path=folder, checkpoint_freq=freq, resume=True) if resume else {}


def _result(scores, jains, errors, rewards, training, **extra):
    out = {"scores": scores, "jains": jains, "channel_errors": errors, "average_rewards": rewards,
           "training": training}
    out.update(extra)
    return out


def xp_load(out_dir="combinatorial_load", learner="d2dppo", n_seeds=1, loads=None, num_iter=2000, n_epoch=5,
            n_envs=10, test_freq=100, test_episodes=1000, setup="setup_8_channels", device=None,
            result_name="results/mcappo_8_channels.p", resume=False):
    """xp_load.py: for every load, train on the heterogeneous 8-channel env, reload the best model, test.
    resume=True: every training run checkpoints into its model folder (``_ckpt_kw``) and continues from there."""
    from .envs import CombinatorialEnv
    s = presets.SETUPS[setup]
    loads = s["loads_list"] if loads is None else loads
    _mk(os.path.join(out_dir, "results"))
    gamma = 0.6 if learner == "d2dppo" else 0.4                      # xp_load.py:80 / :95
    scores, jains, errors, rewards, training = [], [], [], [], []
    for seed in range(n_seeds):
        row = [[], [], [], [], []]
        for load in loads:
            folder = _mk(os.path.join(out_dir, f"models_mcappo{s['n_channels']}_seed_{seed}_load_{load}"))
            env = CombinatorialEnv(n_envs=n_envs, device=device, seed=42 + seed,
                                   **presets.combinatorial_kwargs(setup, load=load, homogeneous_size=True))
            if learner == "irdqn":
                # the run the script keeps commented out (xp_load.py:111-131): same settings, idqn.train(20000) and
                # idqn.test(500) scaled by the caller through num_iter / test_episodes; channel errors / rewards are ""
                from .algorithms.irdqn import iRDQN
                idqn = iRDQN(env, history_len=s["n_agents"], replay_start_size=100, replay_buffer_size=100000,
                             gamma=0.4, update_target_frequency=100, minibatch_size=64, learning_rate=1e-4,
                             update_frequency=1, initial_exploration_rate=1, final_exploration_rate=0.1,
                             adam_epsilon=1e-8, loss="huber", seed=seed)
                res = idqn.train(num_iter, **_ckpt_kw(resume, folder, test_freq))
                score, jain = idqn.test(test_episodes)
                for lst, v in zip(row, (score, jain, "", "", res)):
                    lst.append(v)
                continue
            ppo = _learner(learner, env, folder, seed, hidden_size=64, gamma=gamma, policy_lr=3e-4, value_lr=1e-3,
                           useRNN=True, combinatorial=True, history_len=s["n_agents"], early_stopping=True)
            res = ppo.train(num_iter=num_iter, n_epoch=n_epoch, num_episodes=n_envs, test_freq=test_freq,
                            **_ckpt_kw(resume, folder, test_freq))
            if os.path.exists(os.path.join(folder, "agent_0.pth")):
                ppo.load(folder)
            out = ppo.test(test_episodes)
            for lst, v in zip(row, (*out, res)):
                lst.append(v)
        scores.append(np.array(row[0])), jains.append(np.array(row[1])), errors.append(np.array(row[2]))
        rewards.append(np.array(row[3])), training.append(row[4])
    result = _result(scores, jains, errors, rewards, training)
    with open(os.path.join(out_dir, result_name), "wb") as f:
        pickle.dump(result, f)
    return result


def xp_n_agents(out_dir="xp_3gpp_homogeneous", learner="random_access", n_seeds=1, n_agents_list=(4, 8, 12, 16),
                load=1 / 14, n_envs=500, cv_episodes=50, test_episodes=500, num_iter=2000, n_epoch=5, test_freq=100,
                device=None, result_name="results/aloha.p", resume=False):
    """xp_n_agents.py: N-agent sweep on 4 channels; the active block of the script is the random-access baseline
    with its transmission probability picked by ``get_best_transmission_probs`` (:137-140).  resume=True: the learner
    runs checkpoint into their model folders and continue from there (the baseline has no training state)."""
    from .algorithms.baselines import CombinatorialRandomAccess
    from .envs import CombinatorialEnv
    _mk(os.path.join(out_dir, "results"))
    scores, jains, errors, rewards, training = [], [], [], [], []
    for seed in range(n_seeds):
        row = [[], [], [], [], []]
        for n_agents in n_agents_list:
            env = CombinatorialEnv(n_envs=n_envs, device=device, seed=42 + seed,
                                   **presets.n_agents_sweep_kwargs(n_agents, load=load))
            if learner == "random_access":
                gf = CombinatorialRandomAccess(env)
                cv = gf.get_best_transmission_probs(cv_episodes)
                gf.transmission_prob = gf.transmission_prob_list[int(np.argmax(cv))]
                out, res = gf.run(test_episodes), None
            else:
                folder = _mk(os.path.join(out_dir, f"models_mcappo_seed_{seed}_k_{n_agents}"))
                ppo = _learner(learner, env, folder, seed, hidden_size=64, gamma=0.6 if learner == "d2dppo" else 0.4,
                               policy_lr=3e-4, value_lr=1e-3, useRNN=True, combinatorial=True,
                               history_len=min(n_agents, 10), early_stopping=True)
                res = ppo.train(num_iter=num_iter, n_epoch=n_epoch, num_episodes=n_envs, test_freq=test_freq,
                                **_ckpt_kw(resume, folder, test_freq))
                out = ppo.test(test_episodes)
            for lst, v in zip(row, (*out, res)):
                lst.append(v)
        scores.append(np.array(row[0])), jains.append(np.array(row[1])), errors.append(np.array(row[2]))
        rewards.append(np.array(row[3])), training.append(row[4])
    result = _result(scores, jains, errors, rewards, training if learner != "random_access" else [],
                     xp_params={"n_agents": list(n_agents_list), "deadlines": 7})
    with open(os.path.join(out_dir, result_name), "wb") as f:
        pickle.dump(result, f)
    return result


def run_ma_baselines(out_dir="combinatorial_load", n_seeds=1, n_envs=1000, cv_episodes=100, test_episodes=1000,
                     setup="setup", device=None, result_name="results/aloha_16_channels.p"):
    """run_ma_baselines.py: writes setup.p, then the random-access baseline over ``loads_list`` (16 channels, ragged
    observations: ``homogeneous_size`` keeps its default False, :58-69)."""
    from .algorithms.baselines import CombinatorialRandomAccess
    from .envs import CombinatorialEnv
    s = presets.SETUPS[setup]
    _mk(os.path.join(out_dir, "results"))
    presets.write_load_files(out_dir)                                 # run_ma_baselines.py:34
    gf_scores, gf_jains, gf_errors, gf_rewards = [], [], [], []
    for seed in range(n_seeds):
        row = [[], [], [], []]
        for load in s["loads_list"]:
            env = CombinatorialEnv(n_envs=n_envs, device=device, seed=42 + seed,
                                   **presets.combinatorial_kwargs(setup, load=load, homogeneous_size=False))
            gf = CombinatorialRandomAccess(env)
            cv = gf.get_best_transmission_probs(cv_episodes)
            gf.transmission_prob = gf.transmission_prob_list[int(np.argmax(cv))]
            for lst, v in zip(row, gf.run(test_episodes)):
                lst.append(v)
        gf_scores.append(row[0]), gf_jains.append(row[1]), gf_errors.append(row[2]), gf_rewards.append(row[3])
    result = {"gf_scores": gf_scores, "gf_jains": gf_jains, "gf_channel_errors": gf_errors,
              "gf_average_rewards": gf_rewards}
    with open(os.path.join(out_dir, result_name), "wb") as f:
        pickle.dump(result, f)
    return result


def xp_gamma(out_dir=".", gammas=(0.2, 0.4, 0.6, 0.8, 0.99), n_agents=5, n_channels=16, load=1 / 3.5,
             num_iter=1000, n_epoch=4, n_envs=10, test_freq=100, test_episodes=500, device=None,
             result_name="results/xp_gamma_ippo.p"):
    """xp_gamma.py: iPPO (Categorical channel pick, GRU, history 10) on ChannelSelectionEnv for several discounts.
    Note: in the reference snapshot this script stops in ``env.step`` (actions arrive as (N, 1), SURVEY.md section
    8c); here the action vector is (N,) per env and the sweep runs."""
    from .envs import ChannelSelectionEnv
    _mk(os.path.join(out_dir, "results"))
    scores, jains, errors, rewards, training = [], [], [], [], []
    for gamma in gammas:
        env = ChannelSelectionEnv(
            n_agents=n_agents, n_channels=n_channels, deadlines=np.array([7] * n_agents),
            period=np.array([7] * n_agents), lbdas=np.array([load] * n_agents), episode_length=200,
            traffic_model="aperiodic", arrival_probs=np.array([1] * n_agents), periodic_devices=[2, 4],
            offsets=np.array([0, 2, 4, 0, 2][:n_agents]), channel_switch=np.array([0.8] * (n_channels + 1)),
            n_envs=n_envs, device=device, seed=42)
        ippo = _learner("ippo", env, None, 0, hidden_size=64, gamma=gamma, policy_lr=3e-4, value_lr=1e-2, useRNN=True,
                        history_len=10, early_stopping=True)
        res = ippo.train(num_iter=num_iter, n_epoch=n_epoch, num_episodes=n_envs, test_freq=test_freq)
        out = ippo.test(test_episodes)
        for lst, v in zip((scores, jains, errors, rewards, training), (*out, res)):
            lst.append(v)
    result = _result(scores, jains, errors, rewards, training, xp_params={"gammas": list(gammas), "deadlines": 7})
    with open(os.path.join(out_dir, result_name), "wb") as f:
        pickle.dump(result, f)
    return result


def run_ippo_combinatorial(out_dir="combinatorial_load", load=1 / 3, num_iter=2000, n_epoch=5, n_envs=10, test_freq=100,
                           test_episodes=500, device=None, result_name="results/ippo_16_channels.p", resume=False):
    """run_ippo_combinatorial.py:65-94: iPPO (gamma .99, value_lr 1e-2, history 6) on the 16-channel env.
    resume=True: the run checkpoints into its model folder and continues from there."""
    from .envs import CombinatorialEnv
    _mk(os.path.join(out_dir, "results"))
    env = CombinatorialEnv(n_envs=n_envs, device=device, seed=42,
                           **presets.combinatorial_kwargs("setup", load=load, homogeneous_size=True))
    folder = _mk(os.path.join(out_dir, "models_ippo_16"))
    ippo = _learner("ippo", env, folder, 0, hidden_size=64, gamma=0.99, policy_lr=3e-4, value_lr=1e-2, useRNN=True,
                    combinatorial=True, history_len=6, early_stopping=True)
    res = ippo.train(num_iter=num_iter, n_epoch=n_epoch, num_episodes=n_envs, test_freq=test_freq,
                     **_ckpt_kw(resume, folder, test_freq))
    if os.path.exists(os.path.join(folder, "agent_0.pth")):
        ippo.load(folder)                                             # run_ippo_combinatorial.py:93 reloads the best model
    out = ippo.test(test_episodes)
    result = _result([out[0]], [out[1]], [out[2]], [out[3]], [res])
    with open(os.path.join(out_dir, result_name), "wb") as f:
        pickle.dump(result, f)
    return result


# Literal settings of the reference scripts that the drivers above reproduce as their defaults; checked against the
# values parsed from the reference scripts themselves (tests/golden/experiment_constants.json, written by
# oracle/gen_experiment_constants.py; tests/test_presets.py).
DRIVER_CONSTANTS = {
    "xp_load": dict(output_path="combinatorial_load/results/mcappo_8_channels.p", n_seeds=1, hidden_size=64, gamma=0.6,
                    policy_lr=3e-4, value_lr=1e-3, train=dict(num_iter=2000, n_epoch=5, num_episodes=10, test_freq=100),
                    test_episodes=1000),
    "xp_n_agents": dict(output_path="xp_3gpp_homogeneous/results/aloha.p", n_seeds=1, n_channels=4, load=1 / 14,
                        n_agents_list=[4, 8, 12, 16], cv_episodes=50, test_episodes=500),
    "run_ma_baselines": dict(output_path="combinatorial_load/results/aloha_16_channels.p", n_seeds=1, cv_episodes=100,
                             test_episodes=1000),
    "xp_gamma": dict(output_path="results/xp_gamma_ippo.p", n_seeds=1, n_agents=5, n_channels=16, load=1 / 3.5,
                     gammas=[0.2, 0.4, 0.6, 0.8, 0.99], hidden_size=64, policy_lr=3e-4, value_lr=1e-2, history_len=10,
                     train=dict(num_iter=1000, n_epoch=4, num_episodes=10, test_freq=100), test_episodes=500),
    "run_ippo_combinatorial": dict(output_path="combinatorial_load/results/ippo_16_channels.p", n_seeds=1, n_channels=16,
                                   hidden_size=64, gamma=0.99, policy_lr=3e-4, value_lr=1e-2, history_len=6,
                                   train=dict(num_iter=2000, n_epoch=5, num_episodes=10, test_freq=100),
                                   test_episodes=500),
}


def driver_defaults(name):
    """The same settings read back from the driver's signature / body defaults (what a call without arguments runs)."""
    import inspect
    sig = {k: v.default for k, v in inspect.signature(globals()[name]).parameters.items()}
    out = {"output_path": os.path.normpath(os.path.join(sig["out_dir"], sig["result_name"])), "n_seeds": sig.get("n_seeds", 1)}
    for k in ("load", "n_agents", "n_channels", "cv_episodes", "test_episodes"):
        if k in sig:
            out[k] = sig[k]
    if "gammas" in sig:
        out["gammas"] = list(sig["gammas"])
    if "n_agents_list" in sig:
        out["n_agents_list"] = list(sig["n_agents_list"])
    if "num_iter" in sig and name not in ("xp_n_agents",):
        out["train"] = dict(num_iter=sig["num_iter"], n_epoch=sig["n_epoch"], num_episodes=sig["n_envs"],
                            test_freq=sig["test_freq"])
    return out


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("experiment", choices=["xp_load", "xp_n_agents", "run_ma_baselines", "xp_gamma",
                                           "run_ippo_combinatorial"])
    ap.add_argument("--out", default=None)
    ap.add_argument("--learner", default=None)
    ap.add_argument("--num-iter", type=int, default=None)
    ap.add_argument("--n-envs", type=int, default=None)
    ap.add_argument("--test-episodes", type=int, default=None)
    ap.add_argument("--resume", action="store_true", default=None,
                    help="checkpoint every training run into its model folder and continue from there")
    a = ap.parse_args(argv)
    kw = {k: v for k, v in (("out_dir", a.out), ("learner", a.learner), ("num_iter", a.num_iter), ("n_envs", a.n_envs),
                            ("test_episodes", a.test_episodes), ("resume", a.resume)) if v is not None}
    fn = globals()[a.experiment]
    import inspect
    if a.resume and "resume" not in inspect.signature(fn).parameters:
        ap.error(f"--resume: {a.experiment} keeps no training state to resume")
    kw = {k: v for k, v in kw.items() if k in inspect.signature(fn).parameters}
    res = fn(**kw)
    print({k: (v if k != "training" else "...") for k, v in res.items()})


if __name__ == "__main__":
    main()
