"""get_dataset's policies and the benchmark baseline controllers, pinned to the UNMODIFIED reference.

tests/golden/policy_forced.npz (stored in parts) holds, per env x quality, transitions of the reference's own get_dataset run
(chemical_reactor.py:324-420, power_grid.py:194-249, robot_assembly.py:246-308): the observation the policy saw, every
random value it drew (coin, normals / scale, uniforms / half-range -- recorded by interposing np.random.*) and the action
the dataset stores. tests/golden/baseline_agents.npz holds action sequences of the reference's
benchmarks/baseline_agents.py classes (loaded by file path). Generator: tests/golden/make_golden.py policy baselines.

CPU (not gpu): the oracle's policy restatement and the host mirror of the agents against those vectors.
GPU: the device code (Env::policy_ctrl_from / policy_baseline through nig_selftest_policy) against the same vectors.

Tolerances (the contract):
  * which branch a transition takes (coin vs p_ctrl): exact -- a wrong branch shows as an O(1) action error.
  * stored action: |diff| <= 2.5e-7 + 2 ulp. The reference computes sigma * N(0,1) as one float64 draw N(0, sigma) and
    rounds once; the spec multiplies an fp32 standard normal by an fp32 sigma (<= 1 ulp of the noise term each). The
    deterministic parts (controller terms, robot float64 P-control, clips) are bit-exact: checked where no noise enters.
  * baseline controllers: float64 arithmetic like numpy's -> host mirror bit-exact (float64); device action ==
    float32(reference action) bit-exact.
"""
import ctypes as C
import os

import numpy as np
import pytest

from util import ENV_IDS, KINDS, assert_bits_equal, load_golden, ulp_diff

ENV_CLASS = {"reactor": "ChemicalReactorEnv", "grid": "PowerGridEnv", "robot": "RobotAssemblyEnv"}
CASES = [(n, q) for n in ("reactor", "grid", "robot") for q in ("expert", "medium", "mixed", "random")]


def _case(golden_dir, name, quality):
    g = load_golden(golden_dir, "policy_forced")
    key = f"{name}_{quality}"
    coin = g[key + "_coin"]
    coin32 = np.where(np.isfinite(coin), coin, 0.5).astype(np.float32)
    return g[key + "_obs"], coin32, g[key + "_z"], g[key + "_u"], g[key + "_action"]


def _policy_params(name, quality):
    import neorl_industrial as ni
    return getattr(ni, ENV_CLASS[name]).dataset_policy(quality)


def _check_actions(name, quality, got, obs, coin, z, u, want, pp):
    assert got.shape == want.shape and got.dtype == np.float32
    err = np.abs(got.astype(np.float64) - want.astype(np.float64))
    ulps = ulp_diff(got, want)
    ok = (err <= 2.5e-7) | (ulps <= 2)
    assert ok.all(), (name, quality, float(err.max()), int(ulps.max()), np.argwhere(~ok)[:3].tolist())
    # the deterministic parts are bit-exact: rows / columns that no random value enters
    if quality == "expert" and name in ("grid", "robot"):
        assert_bits_equal(got, want, f"{name} expert policy (no random input)")
    if name == "robot":
        ctrl = coin <= pp.p_ctrl
        assert_bits_equal(got[ctrl][:, :3], want[ctrl][:, :3], "robot float64 P-control of the end-effector error")
    if name == "grid" and quality in ("medium", "mixed"):
        ctrl = coin <= pp.p_ctrl
        assert ctrl.any() and (~ctrl).any()
        assert_bits_equal(got[ctrl], want[ctrl], "grid frequency controller branch")


@pytest.mark.parametrize("name,quality", CASES)
def test_oracle_policy_vs_reference_get_dataset(golden_dir, name, quality):
    from oracle import oracle as O
    obs, coin, z, u, want = _case(golden_dir, name, quality)
    _, _, policy, pp = _policy_params(name, quality)
    got = O.policy_forced(KINDS[name], O.copy_policy_params(pp), obs, coin, z, u)
    _check_actions(name, quality, got, obs, coin, z, u, want, pp)


def test_policy_golden_covers_every_branch(golden_dir):
    g = load_golden(golden_dir, "policy_forced")
    for name, quality in CASES:
        key = f"{name}_{quality}"
        assert len(g[key + "_obs"]) >= 300, key
        coin = g[key + "_coin"]
        if quality in ("medium", "mixed"):
            _, _, _, pp = _policy_params(name, quality)
            frac = np.mean(coin < pp.p_ctrl)
            assert np.isfinite(coin).all() and abs(frac - pp.p_ctrl) < 0.06, (key, frac)      # the mix probability itself
        if name == "robot":
            assert np.abs(g[key + "_action"]).max() <= 2.0                                     # robot_assembly.py:289
    assert np.abs(g["grid_random_action"]).max() > 3.0                                          # power_grid.py:223 stores +-5 raw
    assert np.abs(g["reactor_mixed_action"]).max() <= 1.0                                       # chemical_reactor.py:392 clip


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_dataset_sizes_follow_the_reference(golden_dir, name):
    """episode counts / step caps of every quality: n_samples // 1000 episodes (grid, robot), the (episodes, steps) table
    of chemical_reactor.py:333-347; the reference's realised transition counts bound ours (golden stats)."""
    import json
    gold = json.load(open(os.path.join(golden_dir, f"{name}_dataset_stats.json")))
    want_eps = {"reactor": {"expert": 100, "medium": 200, "mixed": 300, "random": 500},
                "grid": {"expert": 100, "medium": 150, "mixed": 200, "random": 80},
                "robot": {"expert": 120, "medium": 180, "mixed": 250, "random": 100}}[name]
    for quality, n_ep in want_eps.items():
        got_ep, n_steps, _, _ = _policy_params(name, quality)
        assert got_ep == n_ep
        assert gold[quality]["n"] <= n_ep * n_steps
        if name != "reactor":
            assert gold[quality]["keys"] == ["actions", "observations", "rewards", "terminals"]


# ---- baseline controllers -------------------------------------------------------------------------------------------
def _agents(name, g):
    from neorl_industrial.benchmarks import ConstantAgent, MPC_Agent, PIDControllerAgent
    S, A = {"reactor": (12, 3), "grid": (32, 8), "robot": (24, 7)}[name]
    kp, ki, kd = g[f"{name}_pid_gains"]
    return {
        "pid": lambda: PIDControllerAgent(S, A, kp=kp, ki=ki, kd=kd, setpoint=g[f"{name}_setpoint"].copy()),
        "pid_default": lambda: PIDControllerAgent(S, A),
        "mpc": lambda: MPC_Agent(S, A),
        "constant": lambda: ConstantAgent(S, A, constant_action=g[f"{name}_constant"].copy()),
    }


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_host_agents_vs_reference_baseline_agents(golden_dir, name):
    g = np.load(os.path.join(golden_dir, "baseline_agents.npz"))
    states = g[f"{name}_states"]
    T, n, _ = states.shape
    for cname, mk in _agents(name, g).items():
        want = g[f"{name}_{cname}_actions"]
        for i in range(0, n, 5):
            agent = mk()
            got = np.stack([np.asarray(agent.act(states[t, i]), np.float64) for t in range(T)])
            assert np.array_equal(got, want[:, i]), (name, cname, i)
    lo, hi, mean, std = g["random_low_high_mean_std"]
    from neorl_industrial.benchmarks import BaselineAgentFactory
    ra = BaselineAgentFactory.create("random", 12, 3, action_low=-0.5, action_high=0.25)
    d = np.array([ra.act(np.zeros(12)) for _ in range(4000)])
    assert d.min() >= -0.5 and d.max() <= 0.25 and abs(d.mean() - mean) < 0.02 and abs(d.std() - std) < 0.02 and lo >= -0.5 and hi <= 0.25


# ---- the device code -------------------------------------------------------------------------------------------------
def _selftest_policy(N, kind, policy, pp, states, coin=None, z=None, u=None):
    states = np.ascontiguousarray(states, np.float32)
    T, n, _ = states.shape
    A = {0: 3, 1: 8, 2: 7}[kind]
    out = np.empty((T, n, A), np.float32)
    ptr = lambda a: None if a is None else np.ascontiguousarray(a, np.float32).ctypes.data_as(C.c_void_p)
    keep = [np.ascontiguousarray(a, np.float32) for a in (coin, z, u) if a is not None]     # noqa: F841 (lifetime)
    N.check(N.lib().nig_selftest_policy(0, kind, policy, C.byref(pp), n, T, ptr(states), ptr(coin), ptr(z), ptr(u),
                                        out.ctypes.data_as(C.c_void_p)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name,quality", CASES)
def test_device_policy_vs_reference_get_dataset(golden_dir, name, quality):
    from neorl_industrial import _native as N
    from oracle import oracle as O
    obs, coin, z, u, want = _case(golden_dir, name, quality)
    _, _, policy, pp = _policy_params(name, quality)
    assert policy == N.POLICY_PCTRL
    got = _selftest_policy(N, KINDS[name], policy, pp, obs[None], coin[None], z[None], u[None])[0]
    _check_actions(name, quality, got, obs, coin, z, u, want, pp)
    assert_bits_equal(got, O.policy_forced(KINDS[name], O.copy_policy_params(pp), obs, coin, z, u), "device vs oracle")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_device_baseline_controllers_vs_reference(golden_dir, name):
    from neorl_industrial import _native as N
    g = np.load(os.path.join(golden_dir, "baseline_agents.npz"))
    states = g[f"{name}_states"]
    for cname, mk in _agents(name, g).items():
        policy, pp = mk().device_policy()
        got = _selftest_policy(N, KINDS[name], policy, pp, states)
        assert_bits_equal(got, g[f"{name}_{cname}_actions"].astype(np.float32), f"{name} {cname}: device vs reference agent")
