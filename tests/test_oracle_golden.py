"""CPU tests: the oracle (oracle/nig_oracle.c) against golden vectors produced by the UNMODIFIED reference
(tests/golden/make_golden.py). This is what pins the oracle; the GPU tests then compare CUDA vs oracle.

Tolerances (written here because they are the contract):
  * every flag, mask, counter: bit-exact.
  * reactor next-state: bit-exact except component 4 (concentration), the only value downstream of exp() within
    a step -- numpy's float32 exp is a SIMD routine that is not correctly rounded, so <= 2 ulp there.
  * reactor reward: |diff| <= 1e-5 * (|reward| + 100*conc') (it contains conc' * 100).
  * grid / robot next-state: bit-exact. Reward: <= 1e-6 relative (numpy's scalar ``x**2`` calls libm powf, which
    is not correctly rounded; everything else is bit-exact).
"""
import os

import numpy as np
import pytest

from oracle import oracle as O
from util import KINDS, assert_bits_equal, load_golden, ulp_diff


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def _check_step_outputs(kind_name, g, ns, r, fl, vm):
    assert_bits_equal((fl & 1) > 0, g["terminated"], "terminated")
    assert_bits_equal((fl & 2) > 0, g["truncated"], "truncated")
    assert_bits_equal((fl & 4) > 0, g["crit"], "critical_shutdown")
    assert_bits_equal(vm, g["viol_mask"], "violation mask")
    ref_r = g["reward"]
    if kind_name == "reactor":
        cols = [c for c in range(12) if c != 4]
        assert_bits_equal(ns[:, cols], g["next_state"][:, cols], "reactor next_state (non-exp columns)")
        assert ulp_diff(ns[:, 4], g["next_state"][:, 4]).max() <= 2
        tol = 1e-5 * (np.abs(ref_r) + 100.0 * np.abs(g["next_state"][:, 4])) + 1e-6
        assert np.all(np.abs(r.astype(np.float64) - ref_r) <= tol)
        # where conc' is bit-identical the reward must be too
        same = ulp_diff(ns[:, 4], g["next_state"][:, 4]) == 0
        assert_bits_equal(r[same], ref_r.astype(np.float32)[same], "reactor reward where conc' matches")
    else:
        assert_bits_equal(ns, g["next_state"], f"{kind_name} next_state")
        assert np.all(np.abs(r.astype(np.float64) - ref_r) <= 1e-6 * np.abs(ref_r) + 1e-6)
        assert np.mean(r == ref_r.astype(np.float32)) > 0.995


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_forced_tuples(golden_dir, name):
    """M independent (state, step counter, action, noise) -> env.step() tuples covering every branch."""
    g = load_golden(golden_dir, f"{name}_forced")
    kind = KINDS[name]
    m = len(g["reward"])
    env = O.OracleEnv(kind, m, auto_reset=False)
    env.state[:] = g["state"]
    env.ep_step[:] = g["ep_step"]
    ns, r, fl, vm = env.step(g["action"], noise=g["noise"] if O.NOISE_DIM[kind] else None)
    _check_step_outputs(name, g, ns, r, fl, vm)
    assert_bits_equal(env.ep_viol, g["n_viol"], "episode violation counter")
    # the golden set must really exercise the logic
    assert g["terminated"].sum() > 100 and g["truncated"].sum() > 50 and g["crit"].sum() > 100


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_trace_replay(golden_dir, name):
    """BASELINE config #1: one env, 1000 random-action steps, reset on done, replayed teacher-forced."""
    g = _load(golden_dir, f"{name}_trace.npz")
    kind = KINDS[name]
    T = len(g["reward"])
    env = O.OracleEnv(kind, 1, auto_reset=True)
    env.reset(init_states=g["state"][:1])
    total_viol = 0
    for t in range(T):
        if name != "reactor":
            assert_bits_equal(env.state[0], g["state"][t], f"state before step {t}")
        assert env.ep_step[0] == g["ep_step"][t]
        ns, r, fl, vm = env.step(g["action"][t:t + 1], noise=g["noise"][t:t + 1] if O.NOISE_DIM[kind] else None,
                                 reset_states=g["reset_state"][t:t + 1])
        assert bool(fl[0] & 1) == g["terminated"][t] and bool(fl[0] & 2) == g["truncated"][t], t
        assert vm[0] == g["viol_mask"][t]
        total_viol += bin(int(vm[0])).count("1")
        assert total_viol == g["total_violations"][t]
        if name == "reactor":
            # free-running inside an episode: exp ulps may accumulate (stated drift tolerance 1e-4 relative)
            np.testing.assert_allclose(ns[0], g["next_state"][t], rtol=1e-4, atol=1e-6)
        else:
            assert_bits_equal(ns[0], g["next_state"][t], f"next_state at step {t}")


def test_robot_spec_trig_vs_reference(golden_dir):
    """RobotAssembly with the project's specified binary64 sin / cos (exp_mode 1 = what the CUDA kernels compute) against
    the reference's outputs (numpy -> libm): flags / masks identical; positions, joints, forces and scores bit-identical
    (the two sin / cos differ by <= 2 ulp of fp64, which does not survive the rounding to fp32); end-effector
    velocities within 1e-12 absolute (a cancelling difference of positions); reward <= 1e-6 relative."""
    g = load_golden(golden_dir, "robot_forced")
    m = len(g["reward"])
    env = O.OracleEnv(O.ROBOT, m, auto_reset=False, exp_mode=1)
    env.state[:] = g["state"]
    env.ep_step[:] = g["ep_step"]
    ns, r, fl, vm = env.step(g["action"])
    assert np.array_equal((fl & 1) != 0, g["terminated"]) and np.array_equal((fl & 2) != 0, g["truncated"])
    assert_bits_equal(vm, g["viol_mask"], "violation mask")
    vel = [14, 15, 16]                       # (pos' - pos) / dt: a cancelling difference, tiny magnitudes amplify fp64 ulps
    rest = [k for k in range(24) if k not in vel]
    assert_bits_equal(ns[:, rest], g["next_state"][:, rest], "positions / joints / forces / scores")
    dv = np.abs(ns[:, vel].astype(np.float64) - g["next_state"][:, vel].astype(np.float64))
    assert np.all(dv <= 1e-12 + 1e-6 * np.abs(g["next_state"][:, vel])), dv.max()
    ref_r = g["reward"].astype(np.float64)
    assert np.all(np.abs(r.astype(np.float64) - ref_r) <= 1e-6 * np.abs(ref_r) + 1e-6)


def test_reactor_freerun_drift(golden_dir):
    """Free-running 500-step episodes (same actions / noise / initial state as the reference run): flags and
    episode lengths identical; state drift <= 1e-3 relative (SURVEY section 7: measured 2e-6 .. 7.5e-5)."""
    g = _load(golden_dir, "reactor_freerun.npz")
    n_ep, T = g["action"].shape[:2]
    for exp_mode in (0, 1):
        env = O.OracleEnv(O.REACTOR, n_ep, auto_reset=False, exp_mode=exp_mode)
        env.reset(init_states=g["init"])
        worst = 0.0
        for t in range(T):
            live = g["length"] > t
            ns, r, fl, vm = env.step(g["action"][:, t], noise=g["noise"][:, t])
            assert_bits_equal((fl & 7)[live], g["flags"][live, t], f"flags at t={t}")
            ref = g["states"][live, t]
            rel = np.abs(ns[live] - ref) / np.maximum(np.abs(ref), 1e-3)
            worst = max(worst, float(rel.max()))
            rr = g["rewards"][live, t]
            assert np.all(np.abs(r[live] - rr) <= 1e-3 * np.abs(rr) + 1e-2)
        assert worst <= 1e-3, worst
        lengths = np.array([np.argmax(env.done_latch[i] > 0) for i in range(n_ep)])
        assert env.done_latch.sum() == (g["length"] < T).sum() + np.sum((g["length"] == T))


def test_spec_exp_accuracy():
    """The fmaf-polynomial exp of the math spec is < 1 ulp from the true value and handles the edges."""
    xs = np.concatenate([np.linspace(-87, 88, 20001), np.linspace(-3, 3, 20001)]).astype(np.float32)
    got = np.array([O.lib().orc_spec_expf(float(x)) for x in xs], np.float32)
    ref = np.exp(xs.astype(np.float64))
    ulp = np.abs(got.astype(np.float64) - ref) / np.spacing(ref.astype(np.float32)).astype(np.float64)
    assert ulp.max() < 1.0
    assert O.lib().orc_spec_expf(100.0) == np.inf and O.lib().orc_spec_expf(-200.0) == 0.0
    assert np.isnan(O.lib().orc_spec_expf(float("nan")))


def test_philox_known_answers():
    """Random123 known-answer vectors for Philox4x32-10 and for Philox4x32-7 (the round count of the spec's streams)."""
    assert O.lib().orc_spec_philox_rounds() == 7
    assert [hex(x) for x in O.philox((0, 0, 0, 0), (0, 0), 7)] == ["0x5f6fb709", "0xd893f64", "0x4f121f81", "0x4f730a48"]
    assert [hex(x) for x in O.philox((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, 7)] == ["0x5207ddc2", "0x45165e59", "0x4d8ee751", "0x8c52f662"]
    assert [hex(x) for x in O.philox((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), 7)] == \
        ["0x4dfccaba", "0x190a87f0", "0xc47362ba", "0xb6b5242a"]
    assert [hex(x) for x in O.philox((0, 0, 0, 0), (0, 0))] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    assert [hex(x) for x in O.philox((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2)] == ["0x408f276d", "0x41c83b0e", "0xa20bc7c6", "0x6d5451fd"]
    assert [hex(x) for x in O.philox((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0))] == \
        ["0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]


def test_spec_normals_are_gaussian():
    z = np.array([O.spec_normals4(3, i, 5, 0, 0) for i in range(40000)]).ravel()
    assert abs(z.mean()) < 0.02 and abs(z.std() - 1) < 0.02
    kurt = ((z - z.mean()) ** 4).mean() / z.var() ** 2
    assert abs(kurt - 3) < 0.1
    assert abs(np.corrcoef(z[0::4], z[1::4])[0, 1]) < 0.03


def test_spec_stream_words_look_uniform_and_independent():
    """Sanity screen of the 7-round streams on the counters the kernels actually use (consecutive env ids x consecutive
    ticks): byte histograms, correlation between neighbouring envs / ticks / words, bit balance, avalanche. (The
    BigCrush evidence for 7 rounds is Salmon et al.; this only guards against a wiring mistake.)"""
    from scipy import stats
    w = O.words_batch(12345, 1000, 512, 77, 256)                    # 131,072 blocks, 524,288 words
    flat = w.reshape(-1)
    for shift in (0, 8, 16, 24):
        hist = np.bincount((flat >> shift) & 0xFF, minlength=256)
        assert stats.chisquare(hist).pvalue > 1e-4, shift
    u = flat.astype(np.float64) / 2.0 ** 32
    assert stats.kstest(u, "uniform").pvalue > 1e-4
    x = w.astype(np.float64)
    for a, b in ((x[:-1, :, 0], x[1:, :, 0]), (x[:, :-1, 0], x[:, 1:, 0]), (x[..., 0], x[..., 1]), (x[..., 2], x[..., 3])):
        assert abs(np.corrcoef(a.ravel(), b.ravel())[0, 1]) < 0.01
    bits = np.unpackbits(flat.view(np.uint8))
    assert abs(bits.mean() - 0.5) < 2e-3
    # avalanche: neighbouring counters differ in about half of their 128 output bits
    d_env = np.unpackbits((w[:-1] ^ w[1:]).view(np.uint8)).mean()
    d_tick = np.unpackbits((w[:, :-1] ^ w[:, 1:]).view(np.uint8)).mean()
    assert abs(d_env - 0.5) < 2e-3 and abs(d_tick - 0.5) < 2e-3


def test_spec_normal_is_the_inverse_cdf():
    """spec_normal(w) == Phi^-1 of the word's probability level to fp32 rounding: the symmetric tail count
    v = 2 (w mod 2^31) + 1 stands for p = v / 2^33, bit 31 is the sign (math spec, DESIGN.md 4). Checked against
    scipy's ndtri over random words, every octave of the tail, and the end points; monotone in the tail count."""
    from scipy.special import ndtri
    from scipy import stats
    rng = np.random.default_rng(11)
    words = np.concatenate([rng.integers(0, 2 ** 32, 200_000, dtype=np.uint64),
                            (rng.integers(0, 2 ** 32, 60_000, dtype=np.uint64) >> rng.integers(1, 31, 60_000).astype(np.uint64)),
                            [0, 1, 2, 3, 2 ** 31 - 1, 2 ** 31, 2 ** 31 + 1, 2 ** 32 - 1]]).astype(np.uint64)
    z = np.array([O.spec_normal(w) for w in words], np.float64)
    v = 2 * (words & np.uint64(0x7FFFFFFF)).astype(np.float64) + 1
    mag = -ndtri(np.float32(v).astype(np.float64) / 2.0 ** 33)          # the spec rounds the count to binary32 first
    ref = np.where(words >> np.uint64(31), -mag, mag)
    np.testing.assert_allclose(z, ref, rtol=0, atol=8e-7)
    assert 6.3 < abs(O.spec_normal(0)) < 6.4 and abs(O.spec_normal(2 ** 31 - 1)) < 1e-6      # deepest tail / centre
    assert O.spec_normal(5) == -O.spec_normal(5 + 2 ** 31)
    order = np.argsort(words[:200_000] & np.uint64(0x7FFFFFFF))
    m = np.abs(z[:200_000])[order]
    assert (np.diff(m) <= 1e-6).all()                                    # |z| falls as the tail count grows
    ks = stats.kstest(z[:200_000], "norm")
    assert ks.pvalue > 1e-3, ks


def test_oracle_auto_reset_and_latch():
    env = O.OracleEnv(O.GRID, 64, auto_reset=True, seed=9)
    env.reset()
    rng = np.random.default_rng(0)
    n_done = 0
    for _ in range(40):
        ns, r, fl, vm = env.step(rng.uniform(-1, 1, (64, 8)).astype(np.float32))
        done = (fl & 3) > 0
        n_done += int(done.sum())
        assert np.all(env.ep_step[done] == 0) and np.all((fl[done] & 8) > 0)
    assert n_done == env.stats[1] and n_done > 64     # grid episodes last ~5 steps under random actions
    env2 = O.OracleEnv(O.GRID, 64, auto_reset=False, seed=9)
    env2.reset()
    for _ in range(40):
        ns, r, fl, vm = env2.step(rng.uniform(-1, 1, (64, 8)).astype(np.float32))
    assert env2.done_latch.all() and np.all(fl == 128) and np.all(r == 0)
