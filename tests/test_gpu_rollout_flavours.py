"""Fused-rollout kernel flavours that only a size, an environment variable, a policy or a constraint set selects: the
two-env packed f32x2 reactor kernel (chosen by default from 131,072 envs per launch, also inside nig_rollout_steps and
nig_rollout_host slices and CUDA graphs), NIG_POLICY_ZERO, the in-kernel baseline controllers with return extrema and
appended bounds, and 64-thread CTAs of the generic kernel; also the default reactor and PowerGrid kernels from
adversarial populations with return extrema. Every result is compared with the CPU oracle (spec-exp mode) bit for bit;
the fp64 statistics to the tolerances of tests/test_gpu_parity.py. A dispatch witness records kernel names so that these
tests cannot lose their target silently when a dispatch threshold moves."""
import numpy as np
import pytest

from util import (KINDS, Track, adversarial, assert_bits_equal, compare_state, compare_stats, kernel_names, set_population,
                  start_pair)

pytestmark = pytest.mark.gpu

PAIR_MIN = 131_072                 # nig_api.cu rollout_range: launches of at least this many reactor envs take the pair kernel


@pytest.fixture(scope="module")
def mods():
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    from oracle import oracle as O
    return ni, N, O, torch


def _compare_window(env, N, tr, ncons, extrema, what):
    counters, sums = env.read_stats()
    compare_stats(N, counters, sums, tr, ncons, extrema, what, env.read_extrema())


def _run_launches(env, orc, tr, N, torch, chunks, policy_id, policy, ncons, extrema, params=None, what=""):
    """One rollout_device launch per chunk against the tracked oracle: per-env outputs, state and the statistics window
    after every launch (then the window restarts on both sides)."""
    n = orc.n
    rsum, vcnt, dcnt = env.empty(), env.empty(dtype=torch.int32), env.empty(dtype=torch.int32)
    for K in chunks:
        env.rollout_device(K, policy_id, params=params, reward_sum=rsum, viol_count=vcnt, done_count=dcnt)
        o_rs, o_v, o_d = tr.launch(K, policy)
        torch.cuda.synchronize()
        w = f"{what} after a {K}-step launch"
        assert_bits_equal(rsum[:n].cpu().numpy(), o_rs, f"{w}: per-env reward sum")
        assert_bits_equal(vcnt[:n].cpu().numpy().astype(np.int64), o_v, f"{w}: per-env violation count")
        assert_bits_equal(dcnt[:n].cpu().numpy().astype(np.int64), o_d, f"{w}: per-env done count")
        compare_state(env, orc, w)
        _compare_window(env, N, tr, ncons, extrema, w)
        env.clear_stats()
        tr.clear()


def _pair_population(O, rng, s0, n, max_steps):
    """The adversarial population in the first 65,536 envs; behind it whole 64-env warps of the pair kernel (32 threads x 2
    envs) with exactly the pair-specific defects: only env 2j outside the invariant, only env 2j + 1, one warp entirely
    outside, and the warp of the unpartnered last env (n odd) spoiled by that env alone."""
    st, ep_step = adversarial(O, O.REACTOR, rng, s0, n, max_steps, clean_from=65_536)
    w0 = 65_536 // 64 + 10
    for q in range(8):                          # eight warps, each with one defect: env 2j of pair j = 5 + q only ...
        st[64 * (w0 + q) + 2 * (5 + q), 8] = 1.0
    w1 = w0 + 16
    for q in range(8):                          # ... and eight with env 2j + 1 of pair j = 11 + q only
        st[64 * (w1 + q) + 2 * (11 + q) + 1, 9] = 0.5
    w2 = w1 + 16
    st[64 * w2:64 * (w2 + 1), 8] = 1.0                                            # a whole warp
    tail = (n - 1) // 64 * 64
    assert (n - 1) % 2 == 0 and tail >= 64 * (w2 + 1)
    st[tail:n] = s0[tail:n]
    ep_step[tail:n] = 0
    st[n - 1, 8] = 1.0                                                            # the partnerless tail env only
    return st, ep_step


# ---------------------------------------------------------------------------------------------------------------------
# 1. the pair kernel at its default dispatch
@pytest.mark.parametrize("max_steps", [None, 60])
@pytest.mark.parametrize("extrema", [False, True])
def test_pair_kernel_default_dispatch_vs_oracle(mods, extrema, max_steps):
    """n = 131,072 + 4,099 reactor envs in one launch take rollout_reactor_pair_kernel; the last thread has no partner. From
    the adversarial population plus the pair-specific defects, four launches (64, 17, 1, 70 steps; a 60-step episode cap
    ends and auto-resets episodes inside the packed loop) == the oracle stepped one tick at a time."""
    ni, N, O, torch = mods
    n = PAIR_MIN + 4_099
    env, orc = start_pair(ni, O, O.REACTOR, n, seed=6060, env_id_offset=1_001, max_episode_steps=max_steps,
                          threads=O.max_threads())
    st, ep_step = _pair_population(O, np.random.default_rng(12), orc.state.copy(), n, env.max_episode_steps)
    set_population(env, orc, st, ep_step)
    env.track_extrema(extrema)
    tr = Track(orc, "reactor")
    _run_launches(env, orc, tr, N, torch, (64, 17, 1, 70), N.POLICY_UNIFORM,
                  lambda: O.policy_actions(orc, O.POLICY_UNIFORM), 3, extrema, what="pair kernel")
    env.close()


# 2. the pair kernel forced at a small size
@pytest.mark.parametrize("block,extrema,auto_reset", [(32, False, True), (32, True, True), (64, False, True),
                                                      (64, True, True), (128, False, True), (128, True, True),
                                                      (32, True, False)])
def test_pair_kernel_forced_small_vs_oracle(mods, monkeypatch, block, extrema, auto_reset):
    """NIG_ROLLOUT_PAIR=1 at 4,096 + 37 envs with 32 / 64 / 128-thread CTAs (32: the one-warp statistics flush with two envs
    per lane). Without auto-reset the dispatcher must fall back to the one-env kernel, with the same results."""
    ni, N, O, torch = mods
    monkeypatch.setenv("NIG_ROLLOUT_PAIR", "1")
    monkeypatch.setenv("NIG_ROLLOUT_BLOCK", str(block))
    n = 4_096 + 37
    env, orc = start_pair(ni, O, O.REACTOR, n, seed=77, env_id_offset=333, max_episode_steps=60, auto_reset=auto_reset)
    rng = np.random.default_rng(block)
    st, ep_step = adversarial(O, O.REACTOR, rng, orc.state.copy(), n, 60)
    st[2 * 700, 8] = 1.0; st[2 * 900 + 1, 9] = 0.5; st[64 * 40:64 * 41, 8] = 1.0
    done = None if auto_reset else (rng.random(n) < 0.05).astype(np.uint8)
    set_population(env, orc, st, ep_step, done)
    env.track_extrema(extrema)
    tr = Track(orc, "reactor")
    _run_launches(env, orc, tr, N, torch, (64, 17, 1, 70), N.POLICY_UNIFORM,
                  lambda: O.policy_actions(orc, O.POLICY_UNIFORM), 3, extrema, what=f"pair kernel, {block} threads")
    env.close()


# 3. the pair kernel inside sliced calls
def test_pair_kernel_in_sliced_device_rollout_vs_oracle(mods):
    """nig_rollout_steps at 1,048,576 - 1,000 envs: 8 slices of 131,072 envs, the first seven take the pair kernel, the
    ragged last one (130,072 envs) the one-env kernel. Two calls of 150 steps in 64-step launches (the second is a graph
    replay): per-env sums in the device's chunked fp32 order, states, counters and statistics == the oracle."""
    ni, N, O, torch = mods
    n, T, K = (1 << 20) - 1_000, 150, 64
    env, orc = start_pair(ni, O, O.REACTOR, n, seed=2027, env_id_offset=5, max_episode_steps=100, threads=O.max_threads())
    tr = Track(orc, "reactor")
    policy = lambda: O.policy_actions(orc, O.POLICY_UNIFORM)
    rsum, vcnt, dcnt = env.empty(), env.empty(dtype=torch.int32), env.empty(dtype=torch.int32)
    for call in range(2):
        env.rollout_steps_device(T, K, N.POLICY_UNIFORM, reward_sum=rsum, viol_count=vcnt, done_count=dcnt)
        total, o_v, o_d = None, np.zeros(n, np.int64), np.zeros(n, np.int64)
        for c0 in range(0, T, K):
            part, v, d = tr.launch(min(K, T - c0), policy)
            total = part if total is None else (total + part).astype(np.float32)
            o_v += v; o_d += d
        torch.cuda.synchronize()
        w = f"sliced call {call}"
        assert_bits_equal(rsum[:n].cpu().numpy(), total, f"{w}: per-env reward sum")
        assert np.array_equal(vcnt[:n].cpu().numpy(), o_v) and np.array_equal(dcnt[:n].cpu().numpy(), o_d), w
        compare_state(env, orc, w)
        _compare_window(env, N, tr, 3, False, w)
        env.clear_stats()
        tr.clear()
    assert env.tick == 2 * T
    env.close()


@pytest.mark.parametrize("direct", [True, False])
def test_pair_kernel_in_host_rollout_vs_oracle(mods, monkeypatch, direct):
    """nig_rollout_host with two slices at 262,144 + 77 envs: slice 0 (131,200 envs) takes the pair kernel, slice 1 the
    one-env kernel; through the direct path (the slices' kernels read / write the page-locked arrays) and the staged one.
    Two calls (the second replays a graph where one is used) == the oracle."""
    ni, N, O, torch = mods
    monkeypatch.setenv("NIG_HOST_SLICES", "2")
    monkeypatch.setenv("NIG_HOST_DIRECT", "3" if direct else "0")
    monkeypatch.setenv("NIG_HOST_DIRECT_MAX_MB", "1e9")
    n, T, K = (1 << 18) + 77, 150, 64
    env, orc = start_pair(ni, O, O.REACTOR, n, seed=88, env_id_offset=3, max_episode_steps=100, threads=O.max_threads())
    tr = Track(orc, "reactor")
    policy = lambda: O.policy_actions(orc, O.POLICY_UNIFORM)
    for call in range(2):
        out = env.rollout_host(T, N.POLICY_UNIFORM, steps_per_launch=K)
        total, o_v, o_d = None, np.zeros(n, np.int64), np.zeros(n, np.int64)
        for c0 in range(0, T, K):
            part, v, d = tr.launch(min(K, T - c0), policy)
            total = part if total is None else (total + part).astype(np.float32)
            o_v += v; o_d += d
        w = f"host call {call}, direct={direct}"
        assert_bits_equal(out["obs"], orc.state, f"{w}: final observations")
        assert_bits_equal(out["reward_sum"], total, f"{w}: per-env reward sum")
        assert np.array_equal(out["violations"], o_v) and np.array_equal(out["episodes"], o_d), w
        compare_state(env, orc, w)
        # the counters / sums a host call returns are the handle's lifetime statistics: the tracker's window spans both calls
        compare_stats(N, out["counters"], out["sums"], tr, 3, False, w)
    env.close()


# 4. the pair kernel under graph capture
@pytest.mark.parametrize("mode", [1, 2])
def test_pair_kernel_graph_replay_vs_eager_and_oracle(mods, mode):
    """test_gpu_graph.py's captured sequence (single steps + a 16-step fused rollout) at 131,072 + 128 reactor envs, so that
    the rollout is the pair kernel: replays == eager stepping, and the final state == the oracle's."""
    ni, N, O, torch = mods
    n = PAIR_MIN + 128
    dev = torch.device("cuda", 0)
    envs = [ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=31) for _ in range(2)]
    graph_env, eager_env = envs
    orc = O.OracleEnv(O.REACTOR, n, seed=31, exp_mode=1, threads=O.max_threads())
    s0 = orc.reset()
    for e in envs:
        assert_bits_equal(e.reset_host(), s0, "reset draw")
    acts = torch.rand((graph_env.A, graph_env.pitch), device=dev) * 2 - 1
    a_host = acts[:, :n].T.contiguous().cpu().numpy()
    bufs = [(e.empty(), e.empty(dtype=torch.uint8), e.empty(dtype=torch.uint8)) for e in envs]

    def body(e, b):
        e.step_device(acts, reward=b[0], flags=b[1], viol_mask=b[2])
        e.step_device(acts, reward=b[0], flags=b[1], viol_mask=b[2])
        e.rollout_device(16, N.POLICY_UNIFORM)
        e.step_device(acts, reward=b[0], flags=b[1], viol_mask=b[2])

    def oracle_body():
        orc.step(a_host, want_next_obs=False)
        orc.step(a_host, want_next_obs=False)
        for _ in range(16):
            orc.step(O.policy_actions(orc, O.POLICY_UNIFORM), want_next_obs=False)
        return orc.step(a_host, want_next_obs=False)[1]

    graph_env.use_device_tick(mode)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        body(graph_env, bufs[0])
    torch.cuda.current_stream().wait_stream(side)
    graph_env.commit_ticks()
    body(eager_env, bufs[1])
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        body(graph_env, bufs[0])
        graph_env.commit_ticks()
    body(eager_env, bufs[1])
    g.replay()
    for _ in range(3):
        g.replay()
        body(eager_env, bufs[1])
    for _ in range(5):
        o_r = oracle_body()
    torch.cuda.synchronize()
    assert graph_env.tick == eager_env.tick == orc.tick == 5 * 19
    sg, stg, vg, dg = graph_env.get_state_host()
    se, ste, ve, de = eager_env.get_state_host()
    assert_bits_equal(sg, se, "state after graph replays vs eager")
    assert np.array_equal(stg, ste) and np.array_equal(vg, ve)
    assert_bits_equal(bufs[0][0][:n].cpu().numpy(), bufs[1][0][:n].cpu().numpy(), "last reward")
    compare_state(eager_env, orc, "eager vs oracle")
    assert_bits_equal(bufs[1][0][:n].cpu().numpy(), o_r, "last reward vs oracle")
    cg, _ = graph_env.read_stats()
    ce, _ = eager_env.read_stats()
    assert cg[:8].tolist() == ce[:8].tolist()
    assert ce[:6].tolist() == orc.stats[:6].tolist()
    graph_env.use_device_tick(False)
    for e in envs:
        e.close()


# 5. dispatch witness
def test_dispatch_witness(mods, monkeypatch):
    """The kernels the tests above and below are written for are the ones that run: recorded by name with torch.profiler."""
    ni, N, O, torch = mods

    def names_of(kind, n, call, **envvars):
        for k, v in envvars.items():
            monkeypatch.setenv(k, v)
        env = ni.NativeEnv(kind, n, device=0, seed=1)
        env.reset_device()
        got = kernel_names(torch, lambda: call(env))
        env.close()
        for k in envvars:
            monkeypatch.delenv(k)
        return got

    def has(names, what):
        return any(what in x for x in names)
    one = lambda e: e.rollout_device(8, N.POLICY_UNIFORM)
    pair = names_of(N.ENV_CHEMICAL_REACTOR, PAIR_MIN + 4_099, one)
    if not pair:
        pytest.skip("torch.profiler recorded no CUDA kernel in this process (no CUPTI activity records)")
    assert has(pair, "rollout_reactor_pair_kernel") and not has(pair, "rollout_kernel"), sorted(pair)
    off = names_of(N.ENV_CHEMICAL_REACTOR, PAIR_MIN + 4_099, one, NIG_ROLLOUT_PAIR="0")
    assert not has(off, "rollout_reactor_pair_kernel") and has(off, "rollout_kernel"), sorted(off)
    sliced = names_of(N.ENV_CHEMICAL_REACTOR, (1 << 20) - 1_000, lambda e: e.rollout_steps_device(64, 64, N.POLICY_UNIFORM))
    assert has(sliced, "rollout_reactor_pair_kernel") and has(sliced, "rollout_kernel"), sorted(sliced)
    grid = names_of(N.ENV_POWER_GRID, 4_133, one)
    assert any("rollout_grid_kernel" in x and "192" in x for x in grid), sorted(grid)
    small = names_of(N.ENV_CHEMICAL_REACTOR, 4_133, one, NIG_ROLLOUT_PAIR="1", NIG_ROLLOUT_BLOCK="32")
    assert has(small, "rollout_reactor_pair_kernel"), sorted(small)


# 6. policies never compared before
def _bound_cons(N, kind):
    from neorl_industrial.vector import make_constraint
    spec = N.env_spec(kind)
    builtins = [make_constraint(N.CON_BUILTIN, cid=k, penalty=spec.constraints[k].penalty, critical=bool(spec.constraints[k].critical))
                for k in range(3)]
    lo, hi = (300.0, 325.0) if kind == 0 else (-0.4, 0.4)
    return builtins + [make_constraint(N.CON_BOUND, si=0, lo=float(np.float32(lo)), hi=float(np.float32(hi)), penalty=-40.0)]


@pytest.mark.parametrize("cons", ["default", "bound1"])
@pytest.mark.parametrize("extrema", [False, True])
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_zero_policy_vs_oracle(mods, name, extrema, cons):
    """NIG_POLICY_ZERO for every env, with and without return extrema, default constraints (CONS_DEFAULT) and one appended
    state bound (the straight-line CONS_BOUNDS1 kernel)."""
    ni, N, O, torch = mods
    kind, n = KINDS[name], 3_000
    cs = None if cons == "default" else _bound_cons(N, kind)
    env, orc = start_pair(ni, O, kind, n, seed=44, env_id_offset=17, max_episode_steps=50, constraints=cs)
    env.track_extrema(extrema)
    tr = Track(orc, name)
    _run_launches(env, orc, tr, N, torch, (70, 33), N.POLICY_ZERO, lambda: O.policy_actions(orc, O.POLICY_ZERO),
                  3 if cs is None else 4, extrema, what=f"zero policy, {cons}")
    env.close()


def test_industrial_env_zero_rollout_vs_oracle(mods):
    """IndustrialEnv.rollout(T, "zero"): host buffers, 64-step launches, one ChemicalReactor-v0 population."""
    ni, N, O, torch = mods
    n, T, K = 1_000, 150, 64
    env = ni.ChemicalReactorEnv(num_envs=n, seed=9, env_id_offset=40, max_episode_steps=60)
    orc = O.OracleEnv(O.REACTOR, n, seed=9, env_id0=40, exp_mode=1, max_episode_steps=60)
    orc.reset()
    res = env.rollout(T, "zero", steps_per_launch=K, reset=True)
    tr = Track(orc, "reactor")
    total, o_v, o_d = None, np.zeros(n, np.int64), np.zeros(n, np.int64)
    for c0 in range(0, T, K):
        part, v, d = tr.launch(min(K, T - c0), lambda: O.policy_actions(orc, O.POLICY_ZERO))
        total = part if total is None else (total + part).astype(np.float32)
        o_v += v; o_d += d
    assert_bits_equal(res["obs"], orc.state, "final state")
    assert_bits_equal(res["reward_sum"], total, "reward_sum")
    assert np.array_equal(res["violations"], o_v) and np.array_equal(res["episodes"], o_d)
    st = res["stats"]
    assert [st["steps"], st["episodes"], st["terminated"], st["truncated"], st["critical_shutdowns"], st["violations"]] == \
        orc.stats[:6].tolist()
    assert (st["successes"], st["episode_length_sum"]) == (tr.succ, tr.len_sum) and st["episodes"] > 0
    np.testing.assert_allclose([st["return_sum"], st["return_sq"]], [tr.ret_sum, tr.ret_sq], rtol=1e-9, atol=1e-6)
    env.close()


@pytest.mark.parametrize("extrema", [False, True])
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_random_baseline_vs_oracle(mods, name, extrema):
    """The in-kernel RandomAgent over an asymmetric range: a = RN(mid + RN(half * u)) with mid = fp32(0.5 (lo + hi)),
    half = fp32(0.5 (hi - lo)) and u the uniform draw of NIG_POLICY_UNIFORM for the same env and tick."""
    ni, N, O, torch = mods
    from neorl_industrial.benchmarks import BaselineAgentFactory
    kind, n = KINDS[name], 3_000
    lo, hi = -0.3, 0.55
    env, orc = start_pair(ni, O, kind, n, seed=13, env_id_offset=9, max_episode_steps=50)
    pid, pp = BaselineAgentFactory.create("random", env.S, env.A, action_low=lo, action_high=hi).device_policy()
    assert pid == N.POLICY_BASELINE and pp.baseline.kind == N.BASELINE_RANDOM
    mid, half = np.float32(0.5 * (lo + hi)), np.float32(0.5 * (hi - lo))

    def policy():
        u = O.policy_actions(orc, O.POLICY_UNIFORM)
        return (mid + (half * u).astype(np.float32)).astype(np.float32)
    env.track_extrema(extrema)
    tr = Track(orc, name)
    _run_launches(env, orc, tr, N, torch, (70, 33), pid, policy, 3, extrema, params=pp, what="random baseline")
    env.close()


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
@pytest.mark.parametrize("kind", ["pid", "mpc"])
def test_pid_mpc_baselines_with_extrema_and_bound_vs_host_agents(mods, name, kind):
    """In-kernel PID / MPC controllers with return extrema tracking and one appended bound (the BASELINE x extrema x
    CONS_BOUNDS1 instantiation) == one host agent per env driving the oracle."""
    ni, N, O, torch = mods
    from neorl_industrial.benchmarks import BaselineAgentFactory as Factory
    ek, n = KINDS[name], 96
    kw = {}
    if kind == "pid":
        sp = {"reactor": [320.0, 253312.0, 50.0], "grid": [0.0] + [1.0] * 7, "robot": [0.3, 0.0, 0.4, 0, 0, 0, 1.0]}[name]
        kw = {"kp": 0.05, "ki": 0.001, "kd": 0.02, "setpoint": np.array(sp, np.float64)}
    cs = _bound_cons(N, ek)
    env, orc = start_pair(ni, O, ek, n, seed=5, env_id_offset=2, max_episode_steps=30, constraints=cs)
    pid, pp = Factory.create(kind, env.S, env.A, **kw).device_policy()
    agents = [Factory.create(kind, env.S, env.A, **kw) for _ in range(n)]
    env.track_extrema(True)
    tr = Track(orc, name)
    policy = lambda: np.stack([ag.act(o) for ag, o in zip(agents, orc.state)]).astype(np.float32)
    _run_launches(env, orc, tr, N, torch, (45, 32), pid, policy, 4, True, params=pp, what=f"{kind} baseline")
    env.close()


# 7. default and opt-in kernel shapes
@pytest.mark.parametrize("extrema", [False, True])
@pytest.mark.parametrize("case", ["reactor_default", "grid_default", "grid_block64", "robot_block64"])
def test_opt_in_shapes_vs_oracle(mods, monkeypatch, case, extrema):
    """The default dispatch of the reactor (rollout_kernel<Reactor>, one-warp CTAs at this size) and of PowerGrid
    (rollout_grid_kernel, 192-thread CTAs), and NIG_ROLLOUT_BLOCK=64 (generic kernel of the grid and the robot), from
    adversarial populations == the oracle."""
    ni, N, O, torch = mods
    name, envvars = {"reactor_default": ("reactor", {}),
                     "grid_default": ("grid", {}),
                     "grid_block64": ("grid", {"NIG_GRID_FAST": "0", "NIG_ROLLOUT_BLOCK": "64"}),
                     "robot_block64": ("robot", {"NIG_ROLLOUT_BLOCK": "64"})}[case]
    for k, v in envvars.items():
        monkeypatch.setenv(k, v)
    kind, n = KINDS[name], 4_096 + 37
    env, orc = start_pair(ni, O, kind, n, seed=21, env_id_offset=96, max_episode_steps=60 if name == "reactor" else None)
    st, ep_step = adversarial(O, kind, np.random.default_rng(kind + 3), orc.state.copy(), n, env.max_episode_steps)
    set_population(env, orc, st, ep_step)
    env.track_extrema(extrema)
    tr = Track(orc, name)
    _run_launches(env, orc, tr, N, torch, (48, 17, 1, 64), N.POLICY_UNIFORM,
                  lambda: O.policy_actions(orc, O.POLICY_UNIFORM), 3, extrema, what=case)
    env.close()
