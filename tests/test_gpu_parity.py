"""GPU parity tests (run with -m gpu on a B200). Everything goes through the C ABI (libnig_b200.so):
CUDA kernels vs (a) the golden vectors produced by the unmodified reference and (b) the CPU oracle.

Contract:
  * vs the oracle in spec-exp mode: EVERYTHING bit-exact (states, rewards, flags, masks, counters, RNG draws),
    teacher-forced and free-running, single-step kernel (all vector widths / layouts) and fused rollout.
  * vs the reference goldens: flags / masks / counters bit-exact; next-state bit-exact except the reactor's
    concentration (downstream of numpy's non-correctly-rounded SIMD exp): <= 2 ulp; rewards within 1e-5 relative
    (reactor, scaled by the conc' term) / 1e-6 relative (grid, robot: libm powf in numpy's scalar x**2).
"""
import os

import numpy as np
import pytest

from util import ENV_IDS, KINDS, assert_bits_equal, load_golden, ulp_diff

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    from oracle import oracle as O
    return ni, N, O, torch


def _native_env(ni, kind, n, **kw):
    return ni.NativeEnv(kind, n, device=0, **kw)


def _wide_states(rng, O, kind, n):
    """Random states that reach every branch (same recipe family as the golden sampler)."""
    S = O.STATE_DIM[kind]
    if kind == O.REACTOR:
        s = np.stack([rng.uniform(300, 360, n), rng.uniform(2e5, 5.3e5, n), rng.uniform(8, 102, n), rng.uniform(4, 52, n),
                      rng.uniform(0, 2, n) * (rng.random(n) < 0.9), rng.uniform(49.9, 100, n), rng.uniform(285, 300, n),
                      rng.uniform(0, 100, n) * (rng.random(n) < 0.5), (rng.random(n) < 0.3) * 1.0, (rng.random(n) < 0.4) * 1.0,
                      rng.uniform(0, 100, n), rng.uniform(0, 51, n)], 1)
    elif kind == O.GRID:
        base = np.array([50, 60, 45, 55, 40, 65, 35, 50], np.float64)
        s = np.concatenate([rng.normal(0, 0.4, (n, 1)), rng.uniform(0.88, 1.12, (n, 8)), base + rng.normal(0, 30, (n, 8)),
                            np.maximum(base + rng.normal(0, 15, (n, 8)), 0), rng.normal(0, 10, (n, 7))], 1)
    else:
        q = rng.uniform(-np.pi, np.pi, (n, 7))
        s = np.concatenate([rng.uniform(-0.7, 0.7, (n, 3)), np.tile([0, 0, 0, 1.0], (n, 1)), q, rng.normal(0, 0.5, (n, 4)),
                            rng.choice([0.0, 10.0, 49.9, 50.0, 79.0, 81.0, -60.0], (n, 3)), rng.uniform(0, 1, (n, 3))], 1)
    assert s.shape == (n, S)
    return s.astype(np.float32)


def _noise(rng, O, kind, n):
    nz = O.NOISE_DIM[kind]
    if nz == 0:
        return None
    sig = {O.REACTOR: [0.1, 500.0], O.GRID: [0.005] * 8 + [1.0] * 8 + [2.0] * 7}[kind]
    return (rng.normal(0, 1, (n, nz)) * np.array(sig)).astype(np.float32)


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_step_vs_reference_goldens(mods, golden_dir, name):
    ni, N, O, torch = mods
    g = load_golden(golden_dir, f"{name}_forced")
    kind, m = KINDS[name], len(g["reward"])
    env = _native_env(ni, kind, m, auto_reset=False)
    env.set_state_host(g["state"], g["ep_step"], np.zeros(m, np.int32), np.zeros(m, np.uint8))
    obs, next_obs, r, fl, vm = env.step_host(g["action"], noise=g["noise"] if env.NZ else None, want_next_obs=True)
    assert_bits_equal((fl & 1) > 0, g["terminated"], "terminated")
    assert_bits_equal((fl & 2) > 0, g["truncated"], "truncated")
    assert_bits_equal((fl & 4) > 0, g["crit"], "critical_shutdown")
    assert_bits_equal(vm, g["viol_mask"], "violation mask")
    if name == "reactor":
        cols = [c for c in range(12) if c != 4]
        assert_bits_equal(next_obs[:, cols], g["next_state"][:, cols], "next_state (non-exp columns)")
        assert ulp_diff(next_obs[:, 4], g["next_state"][:, 4]).max() <= 2
        tol = 1e-5 * (np.abs(g["reward"]) + 100.0 * np.abs(g["next_state"][:, 4])) + 1e-6
        assert np.all(np.abs(r.astype(np.float64) - g["reward"]) <= tol)
    else:
        if name == "robot":
            # FK runs in fp64 with sin/cos from two different libms (numpy's vs CUDA's, both ~1 ulp fp64): after
            # rounding to fp32 nearly every value is bit-identical; the end-effector velocity (pos' - pos) / dt is a
            # cancellation, so there the difference is bounded absolutely (1e-12 of fp64 noise / 0.1) instead.
            ref = g["next_state"]
            assert np.mean(ulp_diff(next_obs, ref) == 0) > 0.999
            vel = [14, 15, 16]
            rest = [c for c in range(24) if c not in vel]
            assert ulp_diff(next_obs[:, rest], ref[:, rest]).max() <= 1
            np.testing.assert_allclose(next_obs[:, vel], ref[:, vel], rtol=1e-5, atol=1e-9)
        else:
            assert_bits_equal(next_obs, g["next_state"], "next_state")
        assert np.all(np.abs(r.astype(np.float64) - g["reward"]) <= 1e-6 * np.abs(g["reward"]) + 1e-5)
    assert_bits_equal(obs, next_obs, "without auto-reset the stored state is s'")
    _, st, vi, dn = env.get_state_host()
    assert_bits_equal(st, g["ep_step"] + 1, "episode step counter")
    assert_bits_equal(vi, g["n_viol"], "episode violation counter")
    assert_bits_equal(dn, g["terminated"] | g["truncated"], "done latch")


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_trace_replay_gym_api(mods, golden_dir, name):
    """BASELINE config #1 through the drop-in gym API: ni.make(id) single env, 1000 steps, reset on done."""
    ni, N, O, torch = mods
    g = np.load(os.path.join(golden_dir, f"{name}_trace.npz"))
    env = ni.make(ENV_IDS[name])
    obs, info = env.reset(options={"init_states": g["state"][:1]})
    assert obs.dtype == np.float32 and obs.shape == (env.state_dim,)
    assert info["step"] == 0 and info["violations"] == 0
    T = len(g["reward"])
    for t in range(T):
        if name != "reactor":
            assert_bits_equal(env.state, g["state"][t], f"state before step {t}")
        obs, r, term, trunc, info = env.step(g["action"][t], noise=g["noise"][t] if env.native.NZ else None)
        assert isinstance(term, bool) and isinstance(trunc, bool) and isinstance(info, dict)
        assert isinstance(r, np.float32 if name == "reactor" else float)
        assert term == bool(g["terminated"][t]) and trunc == bool(g["truncated"][t]), t
        assert info["critical_shutdown"] == bool(g["crit"][t])
        assert info["safety_metrics"].violation_count == g["n_viol"][t]
        assert info["violations"] == g["ep_violations"][t] and info["total_violations"] == g["total_violations"][t]
        assert info["step"] == g["ep_step"][t] + 1
        if name == "reactor":
            np.testing.assert_allclose(obs, g["next_state"][t], rtol=1e-4, atol=1e-6)
            assert abs(float(r) - g["reward"][t]) <= 1e-3 * abs(g["reward"][t]) + 1e-2
        elif name == "grid":
            assert_bits_equal(obs, g["next_state"][t], f"obs at step {t}")
        else:
            assert ulp_diff(obs, g["next_state"][t]).max() <= 1
        if term or trunc:
            with pytest.raises(RuntimeError, match="Environment is done"):
                env.step(g["action"][t])
            env.reset(options={"init_states": g["reset_state"][t:t + 1]})
    env.close()


@pytest.mark.parametrize("name,vec", [("reactor", 1), ("reactor", 2), ("reactor", 4), ("grid", 1), ("robot", 1)])
@pytest.mark.parametrize("layout", ["host_aos", "host_aos_staged", "device_soa"])
def test_step_bitexact_vs_oracle(mods, name, vec, layout, monkeypatch):
    """Teacher-forced single step, every vector width and both layouts, N not a multiple of anything. host_aos: nig_step_host
    runs the kernel in place on the page-locked host arrays (zero-copy, populations up to 131,072 envs); host_aos_staged:
    the same call through device staging buffers and copies (NIG_ZERO_COPY=0, what larger populations get)."""
    ni, N, O, torch = mods
    if layout.startswith("host_aos") and vec != 1:
        pytest.skip("AoS layouts always use VEC=1")
    monkeypatch.setenv("NIG_ZERO_COPY", "0" if layout == "host_aos_staged" else "1")
    if layout == "host_aos_staged":
        layout = "host_aos"
    kind = KINDS[name]
    n = 5003
    rng = np.random.default_rng(10 + kind)
    s0 = _wide_states(rng, O, kind, n)
    steps = rng.integers(0, O.MAX_EPISODE_STEPS[kind], n).astype(np.int32)
    steps[::7] = O.MAX_EPISODE_STEPS[kind] - 1
    a = rng.uniform(-1.5, 1.5, (n, O.ACTION_DIM[kind])).astype(np.float32)
    nz = _noise(rng, O, kind, n)
    rs = _wide_states(rng, O, kind, n)
    monkeypatch.setenv("NIG_STEP_VEC", str(vec))
    for auto_reset in (True, False):
        orc = O.OracleEnv(kind, n, auto_reset=auto_reset, exp_mode=1)
        orc.state[:] = s0
        orc.ep_step[:] = steps
        o_ns, o_r, o_fl, o_vm = orc.step(a, noise=nz, reset_states=rs)
        env = _native_env(ni, kind, n, auto_reset=auto_reset)
        env.set_state_host(s0, steps, np.zeros(n, np.int32), np.zeros(n, np.uint8))
        if layout == "host_aos":
            obs, next_obs, r, fl, vm = env.step_host(a, noise=nz, reset_states=rs, want_next_obs=True)
        else:
            dev = env.torch_device()
            P = env.pitch

            def soa(x):
                t = torch.zeros((x.shape[1], P), dtype=torch.float32, device=dev)
                t[:, :n] = torch.from_numpy(np.ascontiguousarray(x.T)).to(dev)
                return t
            d_obs, d_next = env.empty(env.S), env.empty(env.S)
            d_r, d_fl, d_vm = env.empty(), env.empty(dtype=torch.uint8), env.empty(dtype=torch.uint8)
            env.step_device(soa(a), noise=soa(nz) if nz is not None else None, reset_states=soa(rs), obs=d_obs,
                            next_obs=d_next, reward=d_r, flags=d_fl, viol_mask=d_vm)
            torch.cuda.synchronize()
            obs, next_obs = d_obs[:, :n].T.cpu().numpy(), d_next[:, :n].T.cpu().numpy()
            r, fl, vm = d_r[:n].cpu().numpy(), d_fl[:n].cpu().numpy(), d_vm[:n].cpu().numpy()
            assert_bits_equal(env.state_tensor()[:, :n].T.cpu().numpy(), orc.state, "zero-copy state view")
        assert_bits_equal(fl, o_fl, "flags")
        assert_bits_equal(vm, o_vm, "violation mask")
        assert_bits_equal(next_obs, o_ns, "next_obs")
        assert_bits_equal(r, o_r, "reward")
        assert_bits_equal(obs, orc.state, "state after the call")
        st, es, ev, dn = env.get_state_host()
        assert_bits_equal(st, orc.state, "device state")
        assert_bits_equal(es, orc.ep_step, "ep_step")
        assert_bits_equal(ev, orc.ep_viol, "ep_viol")
        assert_bits_equal(dn, orc.done_latch.astype(bool), "done latch")
        counters, _ = env.read_stats()
        assert counters[:6].tolist() == orc.stats[:6].tolist()
        assert counters[8:11].tolist() == orc.stats[8:11].tolist()
        env.close()


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_free_running_bitexact_vs_oracle(mods, name):
    """In-kernel Philox noise + reset draws vs the oracle's independent restatement of the RNG spec, with
    auto-reset, over many steps; then again without auto-reset (done latch)."""
    ni, N, O, torch = mods
    kind, n = KINDS[name], 777
    T = 450 if name == "reactor" else 120      # reactor episodes last ~370 steps: run long enough to auto-reset
    rng = np.random.default_rng(3)
    for auto_reset in (True, False):
        env = _native_env(ni, kind, n, auto_reset=auto_reset, seed=1234, env_id_offset=5000)
        orc = O.OracleEnv(kind, n, auto_reset=auto_reset, seed=1234, env_id0=5000, exp_mode=1)
        obs0 = env.reset_host()
        assert_bits_equal(obs0, orc.reset(), "reset draw")
        for t in range(T):
            a = rng.uniform(-1, 1, (n, env.A)).astype(np.float32)
            obs, next_obs, r, fl, vm = env.step_host(a, want_next_obs=True)
            o_ns, o_r, o_fl, o_vm = orc.step(a)
            assert_bits_equal(fl, o_fl, f"flags t={t}")
            assert_bits_equal(next_obs, o_ns, f"next_obs t={t}")
            assert_bits_equal(obs, orc.state, f"state t={t}")
            assert_bits_equal(r, o_r, f"reward t={t}")
            assert_bits_equal(vm, o_vm, f"viol t={t}")
        counters, _ = env.read_stats()
        assert counters[:6].tolist() == orc.stats[:6].tolist()
        if auto_reset:
            assert counters[N.ST_EPISODES] > (0 if name == "reactor" else n)
        # masked explicit reset draws fresh (epoch-keyed) states
        mask = (np.arange(n) % 3 == 0).astype(np.uint8)
        assert_bits_equal(env.reset_host(mask=mask), orc.reset(mask=mask), "masked reset")
        env.close()


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
@pytest.mark.parametrize("policy", ["actions_tma", "actions_ldg", "uniform", "pctrl"])
@pytest.mark.parametrize("extrema", [False, True])
def test_rollout_bitexact_vs_oracle(mods, name, policy, extrema):
    """Fused K-step rollout (state in registers) == K oracle steps: final state, counters, per-env sums, stats;
    with nig_track_extrema also the smallest / largest finished-episode return."""
    ni, N, O, torch = mods
    kind, n, K = KINDS[name], 1000, 70      # K not a multiple of the 16-step TMA chunk
    env = _native_env(ni, kind, n, auto_reset=True, seed=77, env_id_offset=128)
    orc = O.OracleEnv(kind, n, auto_reset=True, seed=77, env_id0=128, exp_mode=1)
    env.reset_host(); orc.reset()
    env.track_extrema(extrema)
    dev = env.torch_device()
    rng = np.random.default_rng(5)
    pp = None
    if policy == "pctrl":
        cls = {"reactor": ni.ChemicalReactorEnv, "grid": ni.PowerGridEnv, "robot": ni.RobotAssemblyEnv}[name]
        _, _, _, pp = cls.dataset_policy("mixed")
    rsum, vcnt, dcnt = env.empty(), env.empty(dtype=torch.int32), env.empty(dtype=torch.int32)
    o_rsum = np.zeros(n, np.float32); o_v = np.zeros(n, np.int64); o_d = np.zeros(n, np.int64)
    ep_ret = np.zeros(n, np.float32 if name == "reactor" else np.float64)
    ret_sum = ret_sq = 0.0
    ret_lo, ret_hi = np.inf, -np.inf
    succ = len_sum = 0
    for rep in range(2):                      # two consecutive launches: tick / episode accumulators carry over
        acts = rng.uniform(-1.3, 1.3, (K, n, env.A)).astype(np.float32)
        if policy.startswith("actions"):
            d_act = torch.zeros((K, env.A, env.pitch), dtype=torch.float32, device=dev)
            d_act[:, :, :n] = torch.from_numpy(np.ascontiguousarray(acts.transpose(0, 2, 1))).to(dev)
            env.rollout_device(K, N.POLICY_ACTIONS, actions=d_act, use_tma=(policy == "actions_tma"),
                               reward_sum=rsum, viol_count=vcnt, done_count=dcnt)
        elif policy == "uniform":
            env.rollout_device(K, N.POLICY_UNIFORM, reward_sum=rsum, viol_count=vcnt, done_count=dcnt)
        else:
            env.rollout_device(K, N.POLICY_PCTRL, params=pp, reward_sum=rsum, viol_count=vcnt, done_count=dcnt)
        o_rsum[:] = 0; o_v[:] = 0; o_d[:] = 0
        for t in range(K):
            if policy.startswith("actions"):
                a = acts[t]
            elif policy == "uniform":
                a = O.policy_actions(orc, O.POLICY_UNIFORM)
            else:
                a = O.policy_actions(orc, O.POLICY_PCTRL, O.copy_policy_params(pp))
            steps_before = orc.ep_step.copy()
            ns, r, fl, vm = orc.step(a)
            o_rsum = (o_rsum + r).astype(np.float32)
            ep_ret = (ep_ret + r).astype(ep_ret.dtype) if name == "reactor" else ep_ret + r.astype(np.float64)
            o_v += np.array([bin(int(x)).count("1") for x in vm])
            done = (fl & 3) > 0
            o_d += done
            if done.any():
                er = ep_ret[done].astype(np.float64)
                ret_sum += er.sum(); ret_sq += (er * er).sum(); succ += int((er > 0).sum())
                ret_lo, ret_hi = min(ret_lo, er.min()), max(ret_hi, er.max())
                len_sum += int((steps_before[done] + 1).sum())
                ep_ret[done] = 0
        torch.cuda.synchronize()
        st, es, ev, dn = env.get_state_host()
        assert_bits_equal(st, orc.state, f"state after rollout {rep}")
        assert_bits_equal(es, orc.ep_step, "ep_step")
        assert_bits_equal(ev, orc.ep_viol, "ep_viol")
        if name == "reactor":
            assert_bits_equal(rsum[:n].cpu().numpy(), o_rsum, "per-env reward sum")
        else:   # oracle rewards are rounded to fp32 per step; the kernel sums the same fp32 values
            assert_bits_equal(rsum[:n].cpu().numpy(), o_rsum, "per-env reward sum")
        assert_bits_equal(vcnt[:n].cpu().numpy().astype(np.int64), o_v, "per-env violation count")
        assert_bits_equal(dcnt[:n].cpu().numpy().astype(np.int64), o_d, "per-env done count")
    d = env.stats_dict()
    assert d["steps"] == orc.stats[0] == 2 * K * n
    assert [d["episodes"], d["terminated"], d["truncated"], d["critical_shutdowns"], d["violations"]] == orc.stats[1:6].tolist()
    assert d["violations_per_constraint"] == orc.stats[8:11].tolist()
    assert d["episode_length_sum"] == len_sum and d["successes"] == succ
    if name == "reactor":
        np.testing.assert_allclose(d["return_sum"], ret_sum, rtol=1e-9, atol=1e-6)
        np.testing.assert_allclose(d["return_sq"], ret_sq, rtol=1e-9, atol=1e-6)
    else:     # grid / robot accumulate episode returns in fp64 from unrounded fp64 rewards: tolerance compare
        np.testing.assert_allclose(d["return_sum"], ret_sum, rtol=1e-6, atol=1e-3)
    # return_min / return_max of the finished episodes (utils.py:131-132): order-preserving keys, last fp64 mantissa bit dropped
    lo, hi = env.read_extrema()
    if d["episodes"] == 0 or not extrema:
        assert lo is None and hi is None
    else:
        tol = 1e-15 if name == "reactor" else 1e-6
        np.testing.assert_allclose([lo, hi], [ret_lo, ret_hi], rtol=tol, atol=0 if name == "reactor" else 1e-3)
    env.clear_stats(); torch.cuda.synchronize()
    assert env.read_extrema() == (None, None)
    env.close()


def test_rollout_equals_single_steps(mods):
    """The fused rollout kernel and K single-step launches walk the same trajectory bit-for-bit."""
    ni, N, O, torch = mods
    n, K = 3000, 48
    a = _native_env(ni, 0, n, seed=5)
    b = _native_env(ni, 0, n, seed=5)
    a.reset_host(); b.reset_host()
    dev = a.torch_device()
    acts = torch.rand((K, 3, a.pitch), device=dev) * 2 - 1
    a.rollout_device(K, N.POLICY_ACTIONS, actions=acts, use_tma=True)
    for t in range(K):
        b.step_device(acts[t])
    torch.cuda.synchronize()
    sa, sb = a.get_state_host(), b.get_state_host()
    for x, y, w in zip(sa, sb, ("state", "ep_step", "ep_viol", "done")):
        assert_bits_equal(x, y, w)
    ca, cb = a.read_stats()[0], b.read_stats()[0]
    assert ca[:6].tolist() == cb[:6].tolist() and ca[8:11].tolist() == cb[8:11].tolist()
    assert a.tick == b.tick == K


def test_sharding_invariance(mods):
    """Shards keyed by global env id reproduce the unsharded run bit-for-bit (SURVEY section 8e)."""
    ni, N, O, torch = mods
    n, K = 4096, 64
    whole = _native_env(ni, 1, n, seed=42)
    whole.reset_host()
    whole.rollout_device(K, N.POLICY_UNIFORM)
    torch.cuda.synchronize()
    ref_state = whole.get_state_host()[0]
    ref_stats = whole.read_stats()[0]
    for shards in (2, 4):
        per = n // shards
        states, stats = [], np.zeros(24, np.int64)
        for r in range(shards):
            e = _native_env(ni, 1, per, seed=42, env_id_offset=r * per)
            e.reset_host()
            e.rollout_device(K, N.POLICY_UNIFORM)
            torch.cuda.synchronize()
            states.append(e.get_state_host()[0])
            stats += e.read_stats()[0]
            e.close()
        assert_bits_equal(np.concatenate(states), ref_state, f"{shards} shards")
        assert stats.tolist() == ref_stats.tolist()


def test_constraint_descriptors_vs_oracle(mods):
    """SafetyWrapper-style declarative bounds + host-evaluated masks, evaluated in-kernel == oracle."""
    ni, N, O, torch = mods
    from neorl_industrial.vector import make_constraint
    n = 4099
    rng = np.random.default_rng(8)
    s0 = _wide_states(rng, O, O.REACTOR, n)
    a = rng.uniform(-1.5, 1.5, (n, 3)).astype(np.float32)
    nz = _noise(rng, O, O.REACTOR, n)
    hm = rng.integers(0, 4, n).astype(np.uint8)
    f32 = lambda x: float(np.float32(x))
    native_cons = [
        make_constraint(N.CON_BUILTIN, cid=2, penalty=-25.0),                       # re-ordered built-ins
        make_constraint(N.CON_BOUND, si=0, ai=0, coef=f32(0.1), lo=280.0, hi=320.0, penalty=-100.0),   # README band
        make_constraint(N.CON_BUILTIN, cid=0, penalty=-100.0, critical=True),
        make_constraint(N.CON_BOUND, si=1, lo=f32(1.5e5), hi=f32(4.5e5), penalty=-70.0, critical=True),
        make_constraint(N.CON_HOSTMASK, cid=0, penalty=-7.5),
        make_constraint(N.CON_HOSTMASK, cid=1, penalty=-11.0, critical=True),
    ]
    orc_cons = [O.Con(c.kind, c.id, c.si, c.ai, c.coef, c.lo, c.hi, c.penalty, c.critical) for c in native_cons]
    orc = O.OracleEnv(O.REACTOR, n, auto_reset=False, exp_mode=1, builtin=False, extra_cons=orc_cons)
    orc.state[:] = s0
    o_ns, o_r, o_fl, o_vm = orc.step(a, noise=nz, hostmask=hm)
    env = _native_env(ni, 0, n, auto_reset=False, constraints=native_cons)
    env.set_state_host(s0, np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint8))
    obs, next_obs, r, fl, vm = env.step_host(a, noise=nz, hostmask=hm, want_next_obs=True)
    assert_bits_equal(vm, o_vm, "violation mask")
    assert_bits_equal(fl, o_fl, "flags")
    assert_bits_equal(r, o_r, "reward with penalties in constraint order")
    assert len(set(vm.tolist())) > 20
    counters, _ = env.read_stats()
    assert counters[8:14].tolist() == orc.stats[8:14].tolist()
    with pytest.raises(NotImplementedError):
        env.rollout_device(4, N.POLICY_UNIFORM)      # host-evaluated constraints cannot run in a fused rollout
    env.close()


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
@pytest.mark.parametrize("extras", ["one_bound", "two_bounds", "two_with_action_term", "three_bounds"])
def test_rollout_with_wrapper_bounds_bitexact_vs_oracle(mods, name, extras):
    """Fused rollout of an env whose SafetyWrapper appended declarative bounds == the oracle, bit for bit: one / two pure
    state bounds take the straight-line CONS_BOUNDS1 / 2 kernels, an action term or a third bound the guarded descriptor
    loop (CONS_PREFIX); TMA-staged actions and the extrema flavour fall back to CONS_PREFIX for the same constraint set."""
    ni, N, O, torch = mods
    from neorl_industrial.vector import make_constraint
    kind, n, K = KINDS[name], 3000, 70
    f32 = lambda x: float(np.float32(x))
    spec = N.env_spec(kind)
    builtins = [make_constraint(N.CON_BUILTIN, cid=k, penalty=spec.constraints[k].penalty, critical=bool(spec.constraints[k].critical))
                for k in range(3)]
    lo0, hi0 = (300.0, 325.0) if kind == 0 else (-0.4, 0.4)
    lo1, hi1 = (1.2e5, 3.5e5) if kind == 0 else ((0.97, 1.03) if kind == 1 else (-0.3, 0.3))
    b0 = make_constraint(N.CON_BOUND, si=0, lo=f32(lo0), hi=f32(hi0), penalty=-40.0)
    b1 = make_constraint(N.CON_BOUND, si=1, lo=f32(lo1), hi=f32(hi1), penalty=-15.0, critical=True)
    b0a = make_constraint(N.CON_BOUND, si=0, ai=0, coef=f32(0.1), lo=f32(lo0), hi=f32(hi0), penalty=-40.0)
    b2 = make_constraint(N.CON_BOUND, si=2, lo=f32(-1e3), hi=f32(60.0 if kind == 0 else 1.0), penalty=-5.0)
    cons = builtins + {"one_bound": [b0], "two_bounds": [b0, b1], "two_with_action_term": [b0a, b1], "three_bounds": [b0, b1, b2]}[extras]
    env = _native_env(ni, kind, n, auto_reset=True, seed=31, constraints=cons)
    ocons = [O.Con(c.kind, c.id, c.si, c.ai, c.coef, c.lo, c.hi, c.penalty, c.critical) for c in cons]
    orc = O.OracleEnv(kind, n, auto_reset=True, seed=31, exp_mode=1, builtin=False, extra_cons=ocons)
    assert_bits_equal(env.reset_host(), orc.reset(), "reset")
    dev = env.torch_device()
    rsum = env.empty()
    env.rollout_device(K, N.POLICY_UNIFORM, reward_sum=rsum)
    o_rs = O.rollout(orc, K, O.POLICY_UNIFORM, want_reward_sum=True)
    torch.cuda.synchronize()
    assert_bits_equal(rsum[:n].cpu().numpy(), o_rs, "reward sum with penalties")
    # teacher-forced actions through TMA (falls back to the descriptor loop) and, with extrema tracking, the LDG flavour
    rng = np.random.default_rng(2)
    for use_tma, ext in ((True, False), (False, True)):
        acts = rng.uniform(-1.3, 1.3, (16, n, env.A)).astype(np.float32)
        d_act = torch.zeros((16, env.A, env.pitch), dtype=torch.float32, device=dev)
        d_act[:, :, :n] = torch.from_numpy(np.ascontiguousarray(acts.transpose(0, 2, 1))).to(dev)
        env.track_extrema(ext)
        env.rollout_device(16, N.POLICY_ACTIONS, actions=d_act, use_tma=use_tma)
        for t in range(16):
            orc.step(acts[t], want_next_obs=False)
    env.track_extrema(False)
    torch.cuda.synchronize()
    st, es, ev, dn = env.get_state_host()
    assert_bits_equal(st, orc.state, "state"); assert_bits_equal(es, orc.ep_step, "ep_step"); assert_bits_equal(ev, orc.ep_viol, "ep_viol")
    c, _ = env.read_stats()
    assert c[:6].tolist() == orc.stats[:6].tolist()
    assert c[8:8 + len(cons)].tolist() == orc.stats[8:8 + len(cons)].tolist()
    assert c[8 + 3] > 0                                   # the first appended bound really fired
    env.close()
    # return extrema of a wrapped env: the straight-line flavour == the descriptor loop (forced by a third, never-violated
    # bound with zero penalty, which leaves every reward unchanged)
    if extras == "two_bounds":
        neutral = make_constraint(N.CON_BOUND, si=2, lo=f32(-3e38), hi=f32(3e38), penalty=0.0)
        got = []
        for cs in (cons, cons + [neutral]):
            e2 = _native_env(ni, kind, n, auto_reset=True, seed=31, constraints=cs)
            e2.reset_host(); e2.track_extrema(True)
            e2.rollout_steps_device(600 if kind == 0 else 60, 64, N.POLICY_UNIFORM)
            torch.cuda.synchronize()
            got.append((e2.read_extrema(), e2.stats_dict()["episodes"], e2.stats_dict()["return_sum"]))
            e2.close()
        assert got[0][0] == got[1][0] and got[0][0][0] is not None and got[0][1] == got[1][1] > 0
        np.testing.assert_allclose(got[0][2], got[1][2], rtol=1e-12)


def test_safety_wrapper_api(mods):
    """README.md:126-139: SafetyWrapper(env, constraints=[fn], penalty=-100) with a Python callable and with the
    declarative BoundConstraint give identical results; penalties and violation counts follow base.py:179-183."""
    ni, N, O, torch = mods
    from neorl_industrial.safety import SafetyWrapper, BoundConstraint

    def temperature_constraint(state, action):
        next_temp = state[0] + 0.1 * action[0]
        return 280 <= next_temp <= 320

    e1 = SafetyWrapper(ni.make("ChemicalReactor-v0", seed=3), constraints=[temperature_constraint], penalty=-100)
    e2 = SafetyWrapper(ni.make("ChemicalReactor-v0", seed=3),
                       constraints=[BoundConstraint("temperature_constraint", 0, 280, 320, penalty=-100,
                                                    action_index=0, action_coef=0.1)])
    e0 = ni.make("ChemicalReactor-v0", seed=3)
    o1, _ = e1.reset(); o2, _ = e2.reset(); o0, _ = e0.reset()
    assert_bits_equal(o1, o2, "same seed -> same initial state")
    init = o0.copy()[None]
    init[0, 0] = 320.02        # T + 0.1*a0 straddles the README's 320 K bound -> violated about half the time
    o1, _ = e1.reset(options={"init_states": init}); o2, _ = e2.reset(options={"init_states": init})
    o0, _ = e0.reset(options={"init_states": init})
    assert len(e1.safety_constraints) == 4
    rng = np.random.default_rng(0)
    n_extra = 0
    for t in range(300):
        a = rng.uniform(-1, 1, 3).astype(np.float32)
        r1 = e1.step(a); r2 = e2.step(a); r0 = e0.step(a)
        assert_bits_equal(r1[0], r2[0], "obs"); assert r1[1] == r2[1] and r1[2:4] == r2[2:4]
        assert_bits_equal(r1[0], r0[0], "the wrapper does not change the dynamics")
        v1, v0 = r1[4]["safety_metrics"].violation_count, r0[4]["safety_metrics"].violation_count
        assert r1[4]["safety_metrics"].total_constraints == 4
        if v1 > v0:
            n_extra += 1
            if not r0[4]["critical_shutdown"]:      # (base + penalties) + (-100); the -1000 of a shutdown comes after
                assert np.float32(r0[1] + np.float32(-100.0)) == r1[1]
        if r1[2] or r1[3]:
            break
    assert n_extra > 10
    assert e1.unwrap() is e1.env and len(e1.env.safety_constraints) == 3


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_api_contract(mods, name):
    """Port of the reference's own real-env assertions (tests/test_comprehensive_system.py:24-107, :581-628)."""
    ni, N, O, torch = mods
    env = ni.make(ENV_IDS[name])
    assert env.observation_space.shape == (env.state_dim,) and env.action_space.shape == (env.action_dim,)
    obs, info = env.reset()
    assert obs.shape == (env.state_dim,) and isinstance(info, dict)
    total = 0.0
    for _ in range(100):
        a = env.action_space.sample()
        obs, reward, terminated, truncated, info = env.step(a)
        assert obs.shape == (env.state_dim,)
        assert isinstance(reward, (int, float, np.floating)) and isinstance(terminated, bool) and isinstance(truncated, bool)
        assert hasattr(info["safety_metrics"], "violation_count") and hasattr(info["safety_metrics"], "safety_score")
        total += float(reward)
        if terminated or truncated:
            obs, info = env.reset()
    assert abs(total) < 1e6
    for c in env.safety_constraints:
        assert isinstance(c.check_fn(obs, a), (bool, np.bool_))
    assert isinstance(env.state, np.ndarray) and isinstance(env.current_step, int)
    ck = env.get_state()
    o1 = env.step(np.zeros(env.action_dim, np.float32))
    env.set_state(ck)
    o2 = env.step(np.zeros(env.action_dim, np.float32))
    assert_bits_equal(o1[0], o2[0], "checkpoint/resume reproduces the step (state + RNG position)")
    env.close()


def test_batched_gym_api(mods):
    ni, N, O, torch = mods
    n = 1000
    env = ni.make("PowerGrid-v0", num_envs=n, seed=1)
    obs, info = env.reset()
    assert obs.shape == (n, 32) and obs.dtype == np.float32
    ndone = 0
    for _ in range(30):
        a = np.stack([env.action_space.sample() for _ in range(4)]).repeat(n // 4, 0)
        obs, r, term, trunc, info = env.step(a)
        assert obs.shape == (n, 32) and r.shape == (n,) and term.dtype == bool and trunc.dtype == bool
        ndone += int((term | trunc).sum())
        sm = info["safety_metrics"]
        assert sm.violation_count.shape == (n,) and np.all(sm.safety_score <= 1.0)
        assert info["final_observation"].shape == (n, 32)
    assert ndone > n          # grid episodes last ~5 steps under random actions -> auto-reset is the common case
    assert env.total_violations > 0 and env.current_step.shape == (n,)
    assert env.native.stats_dict()["episodes"] == ndone
    env.close()


def test_full_size_rollout_property(mods):
    """BASELINE config #2 at full size: 65,536 envs x 1,000 steps (15 x K=64 + 40) of the fused kernel against the
    multi-threaded oracle: a checksum of the final state plus every counter must agree exactly."""
    ni, N, O, torch = mods
    n, T, K = 65536, 1000, 64
    env = _native_env(ni, 0, n, seed=2024)
    env.reset_host()
    done = 0
    while done < T:
        k = min(K, T - done)
        env.rollout_device(k, N.POLICY_UNIFORM)
        done += k
    torch.cuda.synchronize()
    st, es, ev, dn = env.get_state_host()
    d = env.stats_dict()
    assert d["steps"] == n * T and env.tick == T
    orc = O.OracleEnv(0, n, seed=2024, exp_mode=1, threads=max(1, O.max_threads()))
    orc.reset()
    O.rollout(orc, T, O.POLICY_UNIFORM)
    assert_bits_equal(st, orc.state, "final state of 65,536 envs after 1,000 free-running steps")
    assert_bits_equal(es, orc.ep_step, "ep_step")
    assert [d["steps"], d["episodes"], d["terminated"], d["truncated"], d["critical_shutdowns"], d["violations"]] == orc.stats[:6].tolist()
    assert d["episodes"] > 100000


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_step_pipelined_kernel_bitexact_vs_oracle(mods, name, monkeypatch):
    """Populations with more tiles than resident CTAs take the persistent TMA-pipelined step kernel (bulk copies into a
    3-stage shared-memory ring); same results as the oracle, bit for bit, including truncation + in-kernel auto-reset,
    a ragged last tile, and the statistics block; and identical to the one-tile-per-CTA kernel. (The reactor and the
    robot are routed to the pipelined kernel -- the grid case checks the large-population dispatch of the plain kernel.)"""
    ni, N, O, torch = mods
    kind = KINDS[name]
    n = 300_007 if name == "reactor" else 160_003
    rng = np.random.default_rng(11)
    finals = []
    for pipe in ("1", "0"):
        monkeypatch.setenv("NIG_STEP_PIPE", pipe)
        env = _native_env(ni, kind, n, auto_reset=True, seed=99, env_id_offset=7)
        orc = O.OracleEnv(kind, n, auto_reset=True, seed=99, env_id0=7, exp_mode=1, threads=8)
        assert_bits_equal(env.reset_host(), orc.reset(), "reset draw")
        # push a third of the envs to the brink of truncation so that the in-kernel reset path runs
        near = np.where(np.arange(n) % 3 == 0, env.max_episode_steps - 2, 0).astype(np.int32)
        env.set_state_host(ep_step=near)
        orc.ep_step[:] = near
        dev = env.torch_device()
        rew, fl, vm = env.empty(), env.empty(dtype=torch.uint8), env.empty(dtype=torch.uint8)
        rng = np.random.default_rng(11)
        for t in range(4):
            a = rng.uniform(-1.2, 1.2, (n, env.A)).astype(np.float32)
            d_a = torch.zeros((env.A, env.pitch), dtype=torch.float32, device=dev)
            d_a[:, :n] = torch.from_numpy(np.ascontiguousarray(a.T)).to(dev)
            env.step_device(d_a, reward=rew, flags=fl, viol_mask=vm)
            torch.cuda.synchronize()
            _, o_r, o_fl, o_vm = orc.step(a, want_next_obs=False)
            assert_bits_equal(fl[:n].cpu().numpy(), o_fl, f"flags t={t} pipe={pipe}")
            assert_bits_equal(rew[:n].cpu().numpy(), o_r, f"reward t={t} pipe={pipe}")
            assert_bits_equal(vm[:n].cpu().numpy(), o_vm, f"viol t={t} pipe={pipe}")
        state, step, viol, done = env.get_state_host()
        assert_bits_equal(state, orc.state, f"state pipe={pipe}")
        assert np.array_equal(step, orc.ep_step) and np.array_equal(viol, orc.ep_viol)
        counters, _ = env.read_stats()
        assert counters[:6].tolist() == orc.stats[:6].tolist()
        assert counters[N.ST_TRUNCATED] > 0 and counters[N.ST_EPISODES] >= counters[N.ST_TRUNCATED]
        finals.append(state.copy())
        env.close()
    assert_bits_equal(finals[0], finals[1], "pipelined vs one-tile-per-CTA kernel")


def test_powergrid_full_size_sharded_property(mods):
    """BASELINE config #3 at full size: PowerGrid-v0, 1,048,576 envs with auto-reset, as one shard and as 8 shards
    keyed by global env id: identical states and counter sums; and two 4,096-env windows of the big run (the first and
    one in the middle of shard 5) equal to the oracle simulating exactly those global ids."""
    ni, N, O, torch = mods
    n, K, shards = 1 << 20, 64, 8
    whole = _native_env(ni, 1, n, seed=314)
    whole.reset_host(want_obs=False)
    whole.rollout_device(K, N.POLICY_UNIFORM)
    whole.rollout_device(K // 2, N.POLICY_UNIFORM)
    torch.cuda.synchronize()
    ref_state, ref_step, ref_viol, _ = whole.get_state_host()
    ref_stats = whole.read_stats()[0].copy()
    whole.close()
    assert ref_stats[N.ST_STEPS] == n * (K + K // 2) and ref_stats[N.ST_EPISODES] > n      # short episodes: everyone reset
    per = n // shards
    stats = np.zeros(24, np.int64)
    for r in range(shards):
        e = _native_env(ni, 1, per, seed=314, env_id_offset=r * per)
        e.reset_host(want_obs=False)
        e.rollout_device(K, N.POLICY_UNIFORM)
        e.rollout_device(K // 2, N.POLICY_UNIFORM)
        torch.cuda.synchronize()
        st, es, ev, _ = e.get_state_host()
        assert_bits_equal(st, ref_state[r * per:(r + 1) * per], f"shard {r} state")
        assert np.array_equal(es, ref_step[r * per:(r + 1) * per]) and np.array_equal(ev, ref_viol[r * per:(r + 1) * per])
        stats += e.read_stats()[0]
        e.close()
    assert stats.tolist() == ref_stats.tolist()          # integer counters: what the NCCL sum all-reduce returns
    for off in (0, 5 * per + 77_777):
        orc = O.OracleEnv(1, 4096, seed=314, env_id0=off, exp_mode=1, threads=8)
        orc.reset()
        O.rollout(orc, K + K // 2, O.POLICY_UNIFORM)
        assert_bits_equal(ref_state[off:off + 4096], orc.state, f"window at global id {off}")
        assert np.array_equal(ref_step[off:off + 4096], orc.ep_step)
