"""nig_rollout_record / NativeEnv.rollout_record_device / TorchIndustrialEnv.rollout: the fused rollout that records every
step into time-major [T, n, ...] device tensors. Recorded rows == the CPU oracle stepped with the same actions, bit for bit
(in-kernel policies, teacher-forced actions and noise; auto-reset on and off); recording changes nothing nig_rollout computes
(state, episode words, per-env sums, statistics, extrema, PID state); baseline and MLP rows replay through nig_step; MLP
actions == nig_selftest_mlp on the recorded observations; field subsets, canaries around every buffer, split calls into offset
views; argument errors; the torch API and its CUDA-graph capture."""
import numpy as np
import pytest

from util import KINDS, assert_bits_equal, popcount8

pytestmark = pytest.mark.gpu

FIELDS = ("obs", "actions", "rewards", "flags", "viol_mask", "terminated", "truncated", "next_obs")


@pytest.fixture(scope="module")
def mods():
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    from oracle import oracle as O
    return ni, N, O, torch


def _shape(env, f, T):
    return (T, env.n, env.A if f == "actions" else env.S) if f in ("obs", "actions", "next_obs") else (T, env.n)


def _dtype(torch, f):
    return torch.float32 if f in ("obs", "actions", "rewards", "next_obs") else torch.uint8


def _alloc(env, torch, T, fields=FIELDS, canary=None):
    """Output tensors; with `canary`, each is the middle of a larger buffer whose 4 KB margins hold the canary value."""
    out, pads = {}, {}
    for f in fields:
        shape, dt = _shape(env, f, T), _dtype(torch, f)
        size = int(np.prod(shape))
        if canary is None:
            out[f] = torch.full(shape, 0x5A, dtype=dt, device=env.torch_device())
        else:
            pad = 4096 // (4 if dt == torch.float32 else 1)
            flat = torch.full((pad + size + pad,), canary, dtype=dt, device=env.torch_device())
            out[f] = flat[pad:pad + size].view(shape)
            pads[f] = (flat, pad, size)
    return out, pads


def _host(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


def _teacher(env, torch, acts):
    """[T, n, A] host actions -> the kernel's [T][A][pitch] device rows."""
    T = acts.shape[0]
    d = torch.zeros((T, acts.shape[2], env.pitch), dtype=torch.float32, device=env.torch_device())
    d[:, :, :env.n] = torch.from_numpy(np.ascontiguousarray(acts.transpose(0, 2, 1))).to(d.device)
    return d


def _compare_rows(got, want, what):
    for f in want:
        if f in got:
            assert_bits_equal(got[f], want[f], f"{what}: {f}")


def _oracle_rows(orc, T, action_fn, noise=None):
    """T oracle steps -> the rows nig_rollout_record writes, and the per-env sums of the launch."""
    rows = {f: [] for f in FIELDS}
    rsum = np.zeros(orc.n, np.float32); vcnt = np.zeros(orc.n, np.int64); dcnt = np.zeros(orc.n, np.int64)
    for t in range(T):
        a = action_fn(t)
        rows["obs"].append(orc.state.copy()); rows["actions"].append(a.copy())
        ns, r, fl, vm = orc.step(a, noise=None if noise is None else noise[t])
        rows["next_obs"].append(ns); rows["rewards"].append(r); rows["flags"].append(fl); rows["viol_mask"].append(vm)
        rows["terminated"].append((fl & 1).astype(np.uint8)); rows["truncated"].append(((fl & 2) >> 1).astype(np.uint8))
        rsum = (rsum + r).astype(np.float32)
        active = (fl & 128) == 0
        vcnt += popcount8(vm)
        dcnt += (active & ((fl & 3) > 0)).astype(np.int64)
    return {f: np.stack(v) for f, v in rows.items()}, rsum, vcnt, dcnt


def _pp(ni, name):
    cls = {"reactor": ni.ChemicalReactorEnv, "grid": ni.PowerGridEnv, "robot": ni.RobotAssemblyEnv}[name]
    return cls.dataset_policy("mixed")[3]


# ---------------------------------------------------------------------------------------------------------------------
# 1. oracle parity
CASES = [(name, pol) for name in ("reactor", "grid", "robot") for pol in ("uniform", "zero", "pctrl", "actions")] + \
        [("reactor", "actions_noise"), ("grid", "actions_noise")]


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("name,policy", CASES)
def test_record_vs_oracle(mods, name, policy, auto_reset):
    """n = 1,000 envs (not a multiple of 128) at env_id_offset 128, two 70-step calls, a 30-step episode cap so that
    episodes end inside the window (auto-reset on: resets; off: NIG_F_INACTIVE rows). Every recorded row, the per-env sums
    and the final state == the oracle, bit for bit."""
    ni, N, O, torch = mods
    kind, n, K = KINDS[name], 1000, 70
    env = ni.NativeEnv(kind, n, device=0, seed=77, env_id_offset=128, max_episode_steps=30, auto_reset=auto_reset)
    orc = O.OracleEnv(kind, n, auto_reset=auto_reset, seed=77, env_id0=128, exp_mode=1, max_episode_steps=30)
    assert_bits_equal(env.reset_host(), orc.reset(), "reset draw")
    rng = np.random.default_rng(kind * 7 + len(policy))
    pp = _pp(ni, name) if policy == "pctrl" else None
    pid = {"uniform": N.POLICY_UNIFORM, "zero": N.POLICY_ZERO, "pctrl": N.POLICY_PCTRL}.get(policy, N.POLICY_ACTIONS)
    rsum, vcnt, dcnt = env.empty(), env.empty(dtype=torch.int32), env.empty(dtype=torch.int32)
    for call in range(2):
        acts = rng.uniform(-1.3, 1.3, (K, n, env.A)).astype(np.float32)
        noise = rng.normal(0, 1, (K, n, env.NZ)).astype(np.float32) if policy == "actions_noise" else None
        d_act = _teacher(env, torch, acts) if pid == N.POLICY_ACTIONS else None
        d_nz = _teacher(env, torch, noise) if noise is not None else None
        out, _ = _alloc(env, torch, K)
        env.rollout_record_device(K, pid, out=out, actions=d_act, noise=d_nz, params=pp, reward_sum=rsum, viol_count=vcnt,
                                  done_count=dcnt)
        if pid == N.POLICY_ACTIONS:
            fn = lambda t: acts[t]
        elif policy == "pctrl":
            fn = lambda t: O.policy_actions(orc, O.POLICY_PCTRL, O.copy_policy_params(pp))
        else:
            fn = lambda t: O.policy_actions(orc, O.POLICY_UNIFORM if policy == "uniform" else O.POLICY_ZERO)
        want, o_rs, o_v, o_d = _oracle_rows(orc, K, fn, noise)
        torch.cuda.synchronize()
        w = f"{name} {policy} auto_reset={auto_reset} call {call}"
        _compare_rows(_host(out), want, w)
        assert_bits_equal(rsum[:n].cpu().numpy(), o_rs, f"{w}: reward_sum")
        assert np.array_equal(vcnt[:n].cpu().numpy(), o_v) and np.array_equal(dcnt[:n].cpu().numpy(), o_d), w
        st, ep_step, ep_viol, done = env.get_state_host()
        assert_bits_equal(st, orc.state, f"{w}: state")
        assert np.array_equal(ep_step, orc.ep_step) and np.array_equal(done, orc.done_latch.astype(bool)), w
        flags = want["flags"]
        if auto_reset:
            assert (flags & 8).any(), f"{w}: no auto-reset inside the window"
        else:
            assert (flags == 128).any(), f"{w}: no inactive rows"
    assert env.tick == 2 * K
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. recording is a side output
def _policy_setup(ni, N, env, name, policy, rng):
    """(policy id, params, teacher-forced action rows) of a policy name; MLP / PID set up on `env`."""
    from neorl_industrial.benchmarks import BaselineAgentFactory
    if policy == "mlp":
        from test_gpu_mlp_policy import make_mlp
        env.set_mlp_policy(make_mlp(ni, np.random.default_rng(3), env.S, env.A, (128, 64)))
        return N.POLICY_MLP, None
    if policy == "pid":
        sp = {"reactor": [320.0, 253312.0, 50.0], "grid": [0.0] + [1.0] * 7, "robot": [0.3, 0.0, 0.4, 0, 0, 0, 1.0]}[name]
        return BaselineAgentFactory.create("pid", env.S, env.A, kp=0.05, ki=0.001, kd=0.02,
                                           setpoint=np.array(sp, np.float64)).device_policy()
    if policy == "pctrl":
        return N.POLICY_PCTRL, _pp(ni, name)
    return {"uniform": N.POLICY_UNIFORM, "zero": N.POLICY_ZERO, "actions": N.POLICY_ACTIONS}[policy], None


@pytest.mark.parametrize("extrema", [False, True])
@pytest.mark.parametrize("policy", ["uniform", "zero", "pctrl", "actions", "pid", "mlp"])
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_record_is_a_side_output(mods, name, policy, extrema):
    """Two handles with the same seed, one running nig_rollout, the other nig_rollout_record with the same descriptors, three
    calls of 70 / 33 / 64 steps (the last with NIG_ROLLOUT_ACCUMULATE): state, episode words, per-env sums, the 24 counters,
    the extrema, the tick and (through the following calls' actions) the PID state are identical; the fp64 sums agree to
    their atomics' order."""
    import ctypes as C
    ni, N, O, torch = mods
    kind, n = KINDS[name], 3_000
    envs = [ni.NativeEnv(kind, n, device=0, seed=99, env_id_offset=5, max_episode_steps=40) for _ in range(2)]
    plain, rec = envs
    rng = np.random.default_rng(1)
    for e in envs:
        e.reset_host()
        e.track_extrema(extrema)
        pid, pp = _policy_setup(ni, N, e, name, policy, rng)
    sums = [(e.empty(), e.empty(dtype=torch.int32), e.empty(dtype=torch.int32)) for e in envs]
    for K, accumulate in ((70, False), (33, False), (64, True)):
        d_act = _teacher(plain, torch, rng.uniform(-1.3, 1.3, (K, n, plain.A)).astype(np.float32)) if pid == N.POLICY_ACTIONS else None
        out, _ = _alloc(rec, torch, K)
        for e, (rs, vc, dc) in zip(envs, sums):            # the same descriptor for both calls
            r = N.Rollout()
            r.n_steps, r.policy, r.flags = K, pid, N.ROLLOUT_ACCUMULATE if accumulate else 0
            r.actions = N.ptr_of(d_act)
            if pp is not None:
                r.pp = pp
            r.reward_sum, r.viol_count, r.done_count = rs.data_ptr(), vc.data_ptr(), dc.data_ptr()
            if e is plain:
                N.check(N.lib().nig_rollout(e._h, C.byref(r), e._stream()))
            else:
                tr = N.Trajectory(*[out[f].data_ptr() for f in FIELDS])
                N.check(N.lib().nig_rollout_record(e._h, C.byref(r), C.byref(tr), e._stream()))
        torch.cuda.synchronize()
        w = f"{name} {policy} extrema={extrema} after {K} steps"
        for a, b in zip(plain.get_state_host(), rec.get_state_host()):
            assert_bits_equal(a, b, f"{w}: state / episode words")
        for a, b in zip(sums[0], sums[1]):
            assert_bits_equal(a[:n].cpu().numpy(), b[:n].cpu().numpy(), f"{w}: per-env sums")
        (c0, s0), (c1, s1) = plain.read_stats(), rec.read_stats()
        assert c0.tolist() == c1.tolist(), w
        # the fp64 sums are added by fp64 atomics of many warps in whatever order they arrive: two nig_rollout runs differ in
        # their last bits just the same
        np.testing.assert_allclose(s1, s0, rtol=1e-12, atol=1e-6, err_msg=f"{w}: fp64 sums")
        assert plain.read_extrema() == rec.read_extrema() and plain.tick == rec.tick, w
    assert c0[N.ST_EPISODES] > 0
    for e in envs:
        e.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. replay through nig_step
@pytest.mark.parametrize("policy", ["pid", "mlp"])
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_replay_through_step(mods, name, policy):
    """The recorded actions stepped through nig_step (AoS, exact-size outputs) on a fresh handle with the same seed reproduce
    every recorded row: the policies the oracle does not implement."""
    ni, N, O, torch = mods
    kind, n, K = KINDS[name], 1000, 70
    rec = ni.NativeEnv(kind, n, device=0, seed=4, env_id_offset=300, max_episode_steps=25)
    rep = ni.NativeEnv(kind, n, device=0, seed=4, env_id_offset=300, max_episode_steps=25)
    assert_bits_equal(rec.reset_host(), rep.reset_host(), "reset draw")
    pid, pp = _policy_setup(ni, N, rec, name, policy, None)
    out, _ = _alloc(rec, torch, K)
    rec.rollout_record_device(K, pid, out=out, params=pp)
    got = _host(out)
    dev = rep.torch_device()
    b = {"obs": torch.empty((n, rep.S), device=dev), "next_obs": torch.empty((n, rep.S), device=dev),
         "rewards": rep.empty(), "flags": rep.empty(dtype=torch.uint8), "viol_mask": rep.empty(dtype=torch.uint8),
         "terminated": rep.empty(dtype=torch.uint8), "truncated": rep.empty(dtype=torch.uint8)}
    obs_prev = rep.get_state_host()[0]
    for t in range(K):
        assert_bits_equal(got["obs"][t], obs_prev, f"{name} {policy} step {t}: obs")
        a = out["actions"][t].contiguous()
        rep.step_device(a, obs=b["obs"], next_obs=b["next_obs"], reward=b["rewards"], flags=b["flags"], viol_mask=b["viol_mask"],
                        terminated=b["terminated"], truncated=b["truncated"], action_layout=N.LAYOUT_AOS, aux_layout=N.LAYOUT_AOS)
        h = {f: v.cpu().numpy() if v.dim() == 2 else v[:n].cpu().numpy() for f, v in b.items()}
        for f in ("next_obs", "rewards", "flags", "viol_mask", "terminated", "truncated"):
            assert_bits_equal(got[f][t], h[f], f"{name} {policy} step {t}: {f}")
        obs_prev = h["obs"]
    assert (got["flags"] & 8).any()
    for e in (rec, rep):
        e.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. MLP actions
@pytest.mark.parametrize("name,hidden", [("reactor", (64, 64)), ("grid", (256, 256)), ("grid", (64,)), ("robot", (128, 256))])
def test_mlp_actions_match_selftest(mods, name, hidden):
    """Recorded MLP actions == nig_selftest_mlp on the recorded observations (same device function, same row in the tile)
    bit for bit, and within fp64_forward's bound of the network; PowerGrid at H = 256 is the shared-memory-tight kernel,
    at H = 64 the one whose staging tile is widened for the transposes."""
    ni, N, O, torch = mods
    from test_gpu_mlp_policy import assert_within, fp64_forward, make_mlp
    kind, n, K = KINDS[name], 1000, 20
    env = ni.NativeEnv(kind, n, device=0, seed=8, env_id_offset=64, max_episode_steps=12)
    env.reset_host()
    pol = make_mlp(ni, np.random.default_rng(11), env.S, env.A, hidden)
    env.set_mlp_policy(pol)
    out, _ = _alloc(env, torch, K, ("obs", "actions", "flags"))
    env.rollout_record_device(K, N.POLICY_MLP, out=out)
    got = _host(out)
    assert (got["flags"] & 8).any()
    obs = got["obs"].reshape(K * n, env.S)
    # nig_selftest_mlp tiles its rows like the rollout: row i of a step keeps its row-in-tile i mod 128 (n is not a multiple
    # of 128, so each step is evaluated on its own)
    st = np.stack([env.selftest_mlp(got["obs"][t]) for t in range(K)])
    assert_bits_equal(got["actions"], st, f"{name} {hidden}: recorded vs selftest actions")
    ref, bound = fp64_forward(pol, obs)
    assert_within(got["actions"].reshape(K * n, env.A), ref, bound, f"{name} {hidden}: vs fp64 forward")
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. field subsets, canaries, split calls
@pytest.mark.parametrize("name,policy", [("reactor", "uniform"), ("grid", "pctrl"), ("robot", "zero"), ("grid", "mlp")])
def test_subsets_canaries_and_split_calls(mods, name, policy):
    """The same run recorded (a) in full with canaries around every buffer, (b) with subsets of the fields NULL, (c) as
    30 + 40 steps into offset views of [70, n, ...] tensors: identical recorded values, no write outside [K][n][dim]."""
    ni, N, O, torch = mods
    kind, n, K = KINDS[name], 1000, 70
    subsets = [FIELDS, ("rewards", "next_obs"), ("obs", "flags", "truncated"), ("actions", "viol_mask", "terminated"), ()]
    runs = []
    for sub in subsets + ["split"]:
        env = ni.NativeEnv(kind, n, device=0, seed=21, env_id_offset=9, max_episode_steps=30)
        env.reset_host()
        pid, pp = _policy_setup(ni, N, env, name, policy, None)
        if sub == "split":
            out, _ = _alloc(env, torch, K)
            for t0, k in ((0, 30), (30, 40)):
                env.rollout_record_device(k, pid, out={f: v[t0:t0 + k] for f, v in out.items()}, params=pp)
        else:
            out, pads = _alloc(env, torch, K, sub, canary=0x7B)
            env.rollout_record_device(K, pid, out=out, params=pp)
            torch.cuda.synchronize()
            for f, (flat, pad, size) in pads.items():
                c = flat.cpu().numpy()
                want = np.array(0x7B, c.dtype)
                assert (c[:pad] == want).all() and (c[pad + size:] == want).all(), f"{name} {f}: write outside the rows"
        torch.cuda.synchronize()
        runs.append((_host(out), env.get_state_host()[0]))
        env.close()
    full, s_full = runs[0]
    for got, s in runs[1:]:
        _compare_rows(got, full, f"{name} {policy}: subset / split")
        assert_bits_equal(s, s_full, f"{name} {policy}: state")


# ---------------------------------------------------------------------------------------------------------------------
# 6. argument errors
def test_argument_errors(mods):
    """Statuses match nig_rollout's for the same descriptor; out == NULL is rejected; the Python checks raise ValueError
    before anything is launched."""
    import ctypes as C
    ni, N, O, torch = mods
    env = ni.NativeEnv(KINDS["reactor"], 300, device=0, seed=1)
    env.reset_host()
    T, dev = 8, env.torch_device()
    nz = torch.zeros((T, env.NZ, env.pitch), device=dev)
    for kw, exc in [(dict(n_steps=0, policy=N.POLICY_UNIFORM), ValueError),
                    (dict(n_steps=T, policy=N.POLICY_MLP), ValueError),                      # no network yet
                    (dict(n_steps=T, policy=N.POLICY_ACTIONS), ValueError),                  # no actions
                    (dict(n_steps=T, policy=N.POLICY_UNIFORM, noise=nz), NotImplementedError),
                    (dict(n_steps=T, policy=17), ValueError)]:
        k = kw.pop("n_steps")
        with pytest.raises(exc):
            env.rollout_device(k, **kw)
        with pytest.raises(exc):
            env.rollout_record_device(k, out={}, **kw)
    env.track_extrema(True)
    acts = torch.zeros((T, env.A, env.pitch), device=dev)
    with pytest.raises(NotImplementedError):
        env.rollout_device(T, N.POLICY_ACTIONS, actions=acts, noise=nz)
    with pytest.raises(NotImplementedError):
        env.rollout_record_device(T, N.POLICY_ACTIONS, actions=acts, noise=nz, out={})
    env.track_extrema(False)
    r = N.Rollout()
    r.n_steps, r.policy = T, N.POLICY_UNIFORM
    assert N.lib().nig_rollout_record(env._h, C.byref(r), None, None) == N.ERR_INVALID
    tick = env.tick
    good, _ = _alloc(env, torch, T)
    bad = [("obs", torch.empty((T, env.n, env.S + 1), device=dev)), ("rewards", torch.empty((T, env.n), dtype=torch.float64, device=dev)),
           ("flags", torch.empty((T, env.n), dtype=torch.bool, device=dev)), ("actions", torch.empty((T, env.n, env.A))),
           ("next_obs", torch.empty((T, env.S, env.n), device=dev).transpose(1, 2)), ("terminated", torch.empty((T + 1, env.n), dtype=torch.bool, device=dev)),
           ("reward", torch.empty((T, env.n), device=dev))]
    for f, x in bad:
        with pytest.raises(ValueError):
            env.rollout_record_device(T, N.POLICY_UNIFORM, out={**good, f: x})
    assert env.tick == tick                                   # nothing launched
    env.rollout_record_device(T, N.POLICY_UNIFORM, out={**good, "terminated": good["terminated"].bool()})
    env.rollout_record_device(T, N.POLICY_ACTIONS, actions=acts, out={}, )     # all fields NULL: behaves like nig_rollout
    assert env.tick == tick + 2 * T
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 7. the torch API
@pytest.mark.parametrize("name", ["reactor", "grid"])
def test_torch_rollout_api(mods, name):
    """TorchIndustrialEnv.rollout: documented keys, shapes and dtypes; a step() afterwards == a handle that stepped the same
    actions with step(); teacher-forced actions are recorded as given."""
    ni, N, O, torch = mods
    from neorl_industrial.torch_env import TorchIndustrialEnv
    from util import ENV_IDS
    n, T = 1000, 50
    a_env = TorchIndustrialEnv(ENV_IDS[name], n, seed=3, max_episode_steps=20)
    b_env = TorchIndustrialEnv(ENV_IDS[name], n, seed=3, max_episode_steps=20)
    a_env.reset(); b_env.reset()
    res = a_env.rollout(T, "random")
    S, A = a_env.state_dim, a_env.action_dim
    want = {"obs": ((T, n, S), torch.float32), "actions": ((T, n, A), torch.float32), "rewards": ((T, n), torch.float32),
            "terminated": ((T, n), torch.bool), "truncated": ((T, n), torch.bool), "final_observation": ((T, n, S), torch.float32),
            "flags": ((T, n), torch.uint8), "violation_mask": ((T, n), torch.uint8)}
    assert set(res) == set(want)
    for k, (shape, dt) in want.items():
        assert tuple(res[k].shape) == shape and res[k].dtype == dt and res[k].device == a_env.device, k
    for t in range(T):
        obs, r, term, trunc, info = b_env.step(res["actions"][t])
        assert_bits_equal(res["rewards"][t].cpu().numpy(), r.cpu().numpy(), f"step {t}: reward")
        assert torch.equal(res["terminated"][t], term) and torch.equal(res["truncated"][t], trunc), t
        assert torch.equal(res["flags"][t], info["flags"]) and torch.equal(res["violation_mask"][t], info["violation_mask"]), t
        assert_bits_equal(res["final_observation"][t].cpu().numpy(), info["final_observation"].cpu().numpy(), f"step {t}")
        if t + 1 < T:
            assert_bits_equal(res["obs"][t + 1].cpu().numpy(), obs.cpu().numpy(), f"step {t}: obs")
    a = torch.rand((n, A), device=a_env.device) * 2 - 1
    oa = a_env.step(a)
    ob = b_env.step(a)
    for x, y in zip(oa[:4], ob[:4]):
        assert torch.equal(x, y)
    acts = torch.rand((T, n, A), device=a_env.device) * 2.4 - 1.2
    res2 = a_env.rollout(T, actions=acts)
    assert torch.equal(res2["actions"], acts)
    for t in range(T):
        ob = b_env.step(acts[t])
        assert torch.equal(res2["rewards"][t], ob[1]) and torch.equal(res2["flags"][t], ob[4]["flags"])
    with pytest.raises(ValueError):
        a_env.rollout(T, "nonsense")
    with pytest.raises(ValueError):
        a_env.rollout(T, out={"rewards": torch.empty((T, n + 1), device=a_env.device)})
    a_env.close(); b_env.close()


def test_torch_rollout_graph_capture(mods):
    """A recording captured in a CUDA graph under device-tick mode 2 with commit_ticks: two replays == two plain calls."""
    ni, N, O, torch = mods
    from neorl_industrial.torch_env import TorchIndustrialEnv
    n, T = 2000, 24
    g_env = TorchIndustrialEnv("ChemicalReactor-v0", n, seed=12, max_episode_steps=30)
    p_env = TorchIndustrialEnv("ChemicalReactor-v0", n, seed=12, max_episode_steps=30)
    g_env.reset(); p_env.reset()
    nat = g_env.native
    nat.use_device_tick(2)
    bufs = g_env.rollout(T, "random")           # first launch and the output tensors outside the capture
    nat.commit_ticks()
    p_env.rollout(T, "random")
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        g_env.rollout(T, "random", out=bufs)
        nat.commit_ticks()
    for rep in range(2):
        g.replay()
        want = p_env.rollout(T, "random")
        torch.cuda.synchronize()
        for k in want:
            assert torch.equal(bufs[k], want[k]), (rep, k)
    nat.use_device_tick(False)
    assert_bits_equal(g_env.native.get_state_host()[0], p_env.native.get_state_host()[0], "state after two replays")
    g_env.close(); p_env.close()
