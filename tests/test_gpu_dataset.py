"""GPU tests of the on-device get_dataset writer and the batched evaluation loops (run with -m gpu)."""
import json
import os
import time

import numpy as np
import pytest

from util import ENV_IDS, KINDS, assert_bits_equal, oracle_dataset

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    from oracle import oracle as O
    return ni, N, O, torch


ENV_CLASS = {"reactor": "ChemicalReactorEnv", "grid": "PowerGridEnv", "robot": "RobotAssemblyEnv"}


@pytest.mark.parametrize("name,quality,n_ep", [("reactor", "mixed", 300), ("reactor", "expert", 100), ("reactor", "random", 200),
                                               ("grid", "mixed", 200), ("grid", "expert", 100), ("robot", "mixed", 250),
                                               ("robot", "expert", 120)])
def test_dataset_bitexact_vs_oracle(mods, name, quality, n_ep):
    ni, N, O, torch = mods
    from neorl_industrial.datasets import generate_dataset_device
    cls = getattr(ni, ENV_CLASS[name])
    _, n_steps, policy, pp = cls.dataset_policy(quality)
    n_steps = min(n_steps, 300)
    incl = name == "reactor"
    env = ni.NativeEnv(KINDS[name], 1, device=0, seed=99, env_id_offset=4096)
    for gen in range(2):            # two consecutive datasets from one handle draw from different derived keys
        dev, m = generate_dataset_device(env, n_ep, n_steps, policy, pp, extensions=True, timeouts=True,
                                         terminals_include_truncation=incl)
        ref, lens = oracle_dataset(O, KINDS[name], n_ep, n_steps, policy, pp, 99, gen, 4096, incl)
        assert m == int(lens.sum()) == len(ref["rewards"])
        for k in ("observations", "actions", "rewards", "next_observations"):
            assert_bits_equal(dev[k].cpu().numpy(), ref[k], f"{k} (dataset {gen})")
        assert_bits_equal(dev["terminals"].cpu().numpy().astype(bool), ref["terminals"], "terminals")
        assert_bits_equal(dev["safety"].cpu().numpy(), ref["safety"], "safety")
        assert not dev["timeouts"].any()
    env.close()


def test_reactor_dataset_layout_and_reference_statistics(mods, golden_dir):
    """Drop-in get_dataset: the reference's keys / dtypes / shapes (chemical_reactor.py:414-420) and, because the RNG
    streams necessarily differ, distributional parity with the reference's own get_dataset runs (goldens)."""
    ni, N, O, torch = mods
    gold = json.load(open(os.path.join(golden_dir, "reactor_dataset_stats.json")))
    env = ni.make("ChemicalReactor-v0", seed=1)
    for quality in ("mixed", "expert", "medium", "random", "anything-else-is-random"):
        d = env.get_dataset(quality)
        g = gold.get(quality, gold["random"])
        assert sorted(d.keys()) == g["keys"]
        n = len(d["rewards"])
        assert d["observations"].shape == (n, 12) and d["observations"].dtype == np.float32
        assert d["actions"].shape == (n, 3) and d["actions"].dtype == np.float32
        assert d["rewards"].dtype == np.float32 and d["terminals"].dtype == bool and d["timeouts"].dtype == bool
        assert not d["timeouts"].any() and np.abs(d["actions"]).max() <= 1.0
        assert abs(n - g["n"]) / g["n"] < 0.12, (quality, n, g["n"])
    # tighter statistics from 10x the reference's episode count
    big = env.get_dataset("mixed", n_episodes=3000)
    g = gold["mixed"]
    n_ep_ref = 300
    assert abs(len(big["rewards"]) / 3000 - g["n"] / n_ep_ref) / (g["n"] / n_ep_ref) < 0.05          # mean episode length
    assert abs(big["terminals"].sum() / 3000 - g["n_terminals"] / n_ep_ref) < 0.08                  # terminal rate
    assert abs(big["rewards"].mean() - g["reward_mean"]) / g["reward_mean"] < 0.10
    np.testing.assert_allclose(big["actions"].mean(0), g["action_mean"], atol=0.03)
    np.testing.assert_allclose(big["actions"].std(0), g["action_std"], atol=0.03)
    np.testing.assert_allclose(big["observations"].mean(0)[[0, 2, 3, 5, 6, 10]], np.array(g["obs_mean"])[[0, 2, 3, 5, 6, 10]], rtol=0.02)
    env.close()


@pytest.mark.parametrize("name", ["grid", "robot"])
def test_other_envs_dataset_contract(mods, name):
    """power_grid.py:244-249 / robot_assembly.py:303-308: four keys, no 'timeouts', unknown quality -> KeyError."""
    ni, N, O, torch = mods
    env = ni.make(ENV_IDS[name], seed=2)
    d = env.get_dataset("mixed", n_episodes=50)
    assert sorted(d.keys()) == ["actions", "observations", "rewards", "terminals"]
    n = len(d["rewards"])
    assert d["observations"].shape == (n, env.state_dim) and d["actions"].shape == (n, env.action_dim)
    assert d["terminals"].dtype == bool and n > 50
    if name == "robot":
        assert np.abs(d["actions"]).max() <= 2.0
    else:
        assert np.abs(d["actions"]).max() > 1.0          # grid stores the unclipped +-3 proposals
    with pytest.raises(KeyError):
        env.get_dataset("no-such-quality")
    env.close()


@pytest.mark.parametrize("name", ["grid", "robot"])
def test_other_envs_dataset_reference_statistics(mods, golden_dir, name):
    """Distributional parity of PowerGrid / RobotAssembly get_dataset with the reference's own runs (goldens from
    power_grid.py:194-249 / robot_assembly.py:246-308, every quality): the RNG streams necessarily differ, so mean episode
    length, termination rate, reward level and the action moments are compared, from 10x the reference's episode count.
    Tolerances are ~3 sigma of the reference sample (80 .. 250 episodes)."""
    ni, N, O, torch = mods
    gold = json.load(open(os.path.join(golden_dir, f"{name}_dataset_stats.json")))
    env = ni.make(ENV_IDS[name], seed=3)
    for quality, g in gold.items():
        n_ep_ref, _, _, _ = type(env).dataset_policy(quality)
        d = env.get_dataset(quality, n_episodes=10 * n_ep_ref)
        n = len(d["rewards"])
        assert d["observations"].dtype == np.float32 and d["actions"].dtype == np.float32 and d["terminals"].dtype == bool
        # an episode either terminates or runs into the 1,000-step cap (a few % of the robot's do, and those few carry most
        # of the transitions: the plain mean length varies 13 .. 54 between reference seeds) -> compare the termination
        # rate and the mean length of the TERMINATED episodes, (n - 1000 * n_capped) / n_terminated
        n_term, n_term_ref = int(d["terminals"].sum()), g["n_terminals"]
        assert abs(n_term / (10 * n_ep_ref) - n_term_ref / n_ep_ref) < 0.08, quality
        len_t = (n - 1000 * (10 * n_ep_ref - n_term)) / n_term
        len_t_ref = (g["n"] - 1000 * (n_ep_ref - n_term_ref)) / n_term_ref
        assert abs(len_t - len_t_ref) / len_t_ref < 0.25, (quality, len_t, len_t_ref)
        # reward level: per-transition rewards are dominated by the -1000 critical-shutdown step that ends most episodes
        # (only where no reference episode ran into the cap: a handful of capped episodes would carry most transitions)
        if n_term_ref == n_ep_ref:
            se = g["reward_std"] / np.sqrt(g["n_terminals"])
            assert abs(d["rewards"].mean() - g["reward_mean"]) < 4 * se + 0.05 * abs(g["reward_mean"]), (quality, d["rewards"].mean(), g["reward_mean"])
        a_std, a_std_ref = d["actions"].std(0), np.array(g["action_std"])
        np.testing.assert_allclose(a_std, a_std_ref, rtol=0.15, atol=0.03, err_msg=quality)
        np.testing.assert_allclose(d["actions"].mean(0), g["action_mean"], atol=0.12 * max(1.0, float(a_std_ref.max())), err_msg=quality)
    env.close()


def test_one_million_transition_dataset(mods):
    """BASELINE config #5: >= 1M 'mixed' ChemicalReactor transitions written on the device in D4RL layout."""
    ni, N, O, torch = mods
    from neorl_industrial.datasets import generate_dataset_device
    _, n_steps, policy, pp = ni.ChemicalReactorEnv.dataset_policy("mixed")
    env = ni.NativeEnv(0, 1, device=0, seed=5)
    n_ep = 3700
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev, m = generate_dataset_device(env, n_ep, n_steps, policy, pp, extensions=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    assert m >= 1_000_000, m
    obs, nxt, term = dev["observations"], dev["next_observations"], dev["terminals"].bool()
    assert torch.isfinite(obs).all() and torch.isfinite(dev["rewards"]).all()
    # structure: inside an episode row i+1 continues row i; an episode starts at batch_time == 0
    starts = obs[:, 11] == 0
    assert int(starts.sum()) == n_ep
    cont = ~starts[1:]
    assert torch.equal(obs[1:][cont], nxt[:-1][cont]), "observations[i+1] must equal next_observations[i] inside an episode"
    assert not term[:-1][cont].any(), "a terminal row must be the last row of its episode"
    assert torch.allclose(obs[:, 11][~starts], nxt[:, 11][:-1][cont])
    print(f"\n1M-transition dataset: {m} transitions in {dt * 1e3:.2f} ms = {m / dt:.3g} transitions/s (incl. length probe + scan)")
    env.close()


def test_evaluate_policy_device_matches_oracle(mods):
    ni, N, O, torch = mods
    from neorl_industrial.rollouts import evaluate_policy_device
    n, T = 2048, 600
    env = ni.make("ChemicalReactor-v0", num_envs=n, seed=21)
    env.reset()
    res = evaluate_policy_device(env, T, N.POLICY_UNIFORM)
    orc = O.OracleEnv(O.REACTOR, n, seed=21, exp_mode=1)
    orc.reset()
    O.rollout(orc, T, O.POLICY_UNIFORM)
    assert res["steps"] == n * T and res["episodes"] == orc.stats[1] > n
    assert res["safety_violations"] == orc.stats[5] and res["emergency_shutdowns"] == orc.stats[4]
    assert res["critical_violations"] == orc.stats[8] + orc.stats[9]
    assert 0.0 <= res["constraint_satisfaction_rate"] <= 1.0 and res["return_std"] > 0
    for k in ("return_mean", "return_std", "length_mean", "length_std", "safety_violations_per_episode", "success_rate",
              "successful_episodes"):
        assert k in res
    assert 100 < res["length_mean"] <= 500
    env.close()


class _PAgent:
    """Minimal trained agent: proportional temperature control (what evaluate_with_safety needs: is_trained + predict)."""
    is_trained = True

    def predict(self, obs, deterministic=True):
        obs = np.atleast_2d(obs)
        a = np.zeros((obs.shape[0], 3), np.float32)
        a[:, 0] = -0.2 * (obs[:, 0] - 320.0) / 50.0
        return a


def test_evaluate_with_safety_single_and_batched(mods):
    ni, N, O, torch = mods
    keys = {"return_mean", "return_std", "return_min", "return_max", "length_mean", "length_std", "safety_violations",
            "safety_violations_per_episode", "critical_violations", "emergency_shutdowns", "constraint_satisfaction_rate",
            "successful_episodes", "success_rate"}
    single = ni.evaluate_with_safety(_PAgent(), ni.make("ChemicalReactor-v0", seed=1), n_episodes=3)
    assert set(single) == keys and single["length_mean"] > 10
    batched = ni.evaluate_with_safety(_PAgent(), ni.make("ChemicalReactor-v0", num_envs=256, seed=1), n_episodes=300)
    assert set(batched) == keys and batched["length_mean"] > 10 and batched["return_max"] >= batched["return_min"]
    with pytest.raises(RuntimeError, match="must be trained"):
        ni.evaluate_with_safety(object(), ni.make("ChemicalReactor-v0"), n_episodes=1)


def test_dataset_n_transitions_target():
    """get_dataset(..., n_transitions=M): whole episodes until at least M rows (BASELINE config 5 asks for 1M rows)."""
    import neorl_industrial as ni
    env = ni.make("ChemicalReactor-v0")
    ds = env.get_dataset("mixed", n_transitions=20_000)
    m = ds["rewards"].shape[0]
    assert 20_000 <= m < 20_000 + 300, m                   # the smallest episode count that reaches M: overshoot < one episode
    assert ds["observations"].shape == (m, 12) and ds["actions"].shape == (m, 3)
    assert ds["terminals"].dtype == bool and ds["timeouts"].dtype == bool and not ds["timeouts"].any()
    assert np.abs(ds["actions"]).max() <= 1.0
    env.close()


def test_reference_timing_harness_keys():
    """neorl_industrial.benchmarks.performance reproduces the env-path sections of performance_benchmark.py."""
    from neorl_industrial.benchmarks import performance as P
    c = P.benchmark_environment_creation(3)
    assert set(c) == {"avg_creation_time", "memory_per_env", "total_time"} and c["avg_creation_time"] > 0
    d = P.benchmark_dataset_loading("medium")
    assert set(d) == {"dataset_size", "load_time", "samples_per_sec"} and d["dataset_size"] > 10_000
    s1 = P.benchmark_environment_steps(200)
    assert set(s1) == {"total_time", "steps_per_sec"} and s1["steps_per_sec"] > 0
    sb = P.benchmark_environment_steps(128, num_envs=4096)
    assert sb["steps_per_sec"] > s1["steps_per_sec"] and sb["num_envs"] == 4096
