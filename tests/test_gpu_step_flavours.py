"""Single-step kernel flavours that only a population size, an environment variable, a constraint set or an argument
layout selects: the persistent TMA-pipelined step_pipe_kernel with appended (CONS_PREFIX) and re-ordered (CONS_GENERIC)
constraint sets, the step_kernel matrix of vector widths x constraint modes with teacher forcing and unpacked
terminated / truncated outputs, the reactor's two-env step kernel at its default dispatch, the persistent kernels under
CUDA-graph capture with the device tick, and the host-step outputs of nig_step_host. Every result is compared with the CPU
oracle (spec-exp mode) bit for bit after every step, the fp64 statistics to the tolerances of
tests/test_gpu_rollout_flavours.py. The dedicated PowerGrid step kernel at its real threshold is
tests/test_gpu_round2.py::test_grid_persistent_step_kernel_from_adversarial_states_and_actions. A dispatch witness records
kernel names so that these tests cannot lose their target silently when a dispatch threshold moves."""
import ctypes as C

import numpy as np
import pytest

from util import KINDS, Track, adversarial, assert_bits_equal, compare_state, compare_stats, kernel_names, template_args

pytestmark = pytest.mark.gpu

# populations clearly above the thresholds of the persistent kernels on a B200 (148 SMs; see the dispatch witness)
GRID_N = 262_147                               # 1,025 tiles of 256 envs: step_grid_kernel<256, 128, 4> from 888 tiles
PIPE_N = {"reactor": 300_007, "robot": 160_003}    # step_pipe_kernel: more tiles than resident CTAs
VEC2_N = 655_363                               # pitch 655,488 >= 2 x 148 x 2048: the reactor's two-env step kernel
CONS_GENERIC, CONS_PREFIX = 0, 2               # nig_kernels.cuh


@pytest.fixture(scope="module")
def mods():
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    from oracle import oracle as O
    return ni, N, O, torch


def _builtins(N, kind, order=(0, 1, 2)):
    from neorl_industrial.vector import make_constraint
    spec = N.env_spec(kind)
    return [make_constraint(N.CON_BUILTIN, cid=k, penalty=spec.constraints[k].penalty,
                            critical=bool(spec.constraints[k].critical)) for k in order]


def _cons(N, kind, which, s0):
    """None (the env's default set, CONS_DEFAULT); "prefix": the built-ins plus two SafetyWrapper bands, a critical one on
    state 1 and one with an action term on state 0 (CONS_PREFIX); "generic": the built-ins re-ordered, a bound and two
    host-mask descriptors (CONS_GENERIC). The bands sit at quantiles of the entry states, so that they fire in a few
    per cent of the envs (the critical one in about 1 %)."""
    from neorl_industrial.vector import make_constraint
    if which == "default":
        return None
    ok = np.isfinite(s0).all(1)

    def q(si, p):
        return float(np.float32(np.quantile(s0[ok, si], p)))
    if which == "prefix":
        return _builtins(N, kind) + [
            make_constraint(N.CON_BOUND, si=1, lo=q(1, 0.005), hi=q(1, 0.995), penalty=-60.0, critical=True),
            make_constraint(N.CON_BOUND, si=0, ai=0, coef=float(np.float32(0.1)), lo=q(0, 0.1), hi=q(0, 0.9), penalty=-15.0)]
    return _builtins(N, kind, (2, 0, 1)) + [
        make_constraint(N.CON_BOUND, si=0, lo=q(0, 0.2), hi=q(0, 0.8), penalty=-40.0),
        make_constraint(N.CON_HOSTMASK, cid=0, penalty=-7.5),
        make_constraint(N.CON_HOSTMASK, cid=1, penalty=-11.0, critical=True)]


def _start(ni, N, O, name, n, *, seed, env_id_offset=0, auto_reset=True, cons="default", population=True):
    """Env and oracle from the same reset draw, then (population=True) the adversarial entry population of
    test_gpu_rollout_flavours.py, and without auto-reset some done latches. Returns env, tracker, number of constraints."""
    kind = KINDS[name]
    probe = O.OracleEnv(kind, n, seed=seed, env_id0=env_id_offset, exp_mode=1, threads=O.max_threads())
    s0 = probe.reset()
    cs = _cons(N, kind, cons, s0)
    env = ni.NativeEnv(kind, n, device=0, seed=seed, env_id_offset=env_id_offset, auto_reset=auto_reset, constraints=cs)
    kw = {} if cs is None else {
        "builtin": False, "extra_cons": [O.Con(c.kind, c.id, c.si, c.ai, c.coef, c.lo, c.hi, c.penalty, c.critical) for c in cs]}
    orc = O.OracleEnv(kind, n, auto_reset=auto_reset, seed=seed, env_id0=env_id_offset, exp_mode=1,
                      threads=O.max_threads(), **kw)
    assert_bits_equal(env.reset_host(), orc.reset(), "reset draw")
    if population:
        rng = np.random.default_rng(seed)
        st, ep_step = adversarial(O, kind, rng, s0, n, env.max_episode_steps)
        ep_step[rng.choice(n, n // 50, replace=False)] = env.max_episode_steps - 1        # truncated on the first step
        done = np.zeros(n, np.uint8) if auto_reset else (rng.random(n) < 0.03).astype(np.uint8)
        env.set_state_host(st, ep_step, np.zeros(n, np.int32), done)
        orc.state[:] = st
        orc.ep_step[:] = ep_step
        orc.ep_viol[:] = 0
        orc.done_latch[:] = done
    return env, Track(orc, name), 3 if cs is None else len(cs)


def _actions(rng, n, A):
    """Over-range actions with NaN / +-inf / -0.0 / far out-of-range components in a few envs."""
    a = rng.uniform(-1.3, 1.3, (n, A)).astype(np.float32)
    i = rng.choice(n, 64, replace=False)
    a[i, rng.integers(0, A, 64)] = rng.choice([np.nan, np.inf, -np.inf, -0.0, 5.0, -7.0], 64).astype(np.float32)
    return a


def _soa(torch, env, x, offset=0):
    """[n, D] host rows -> a [D, pitch] device tensor (the SoA layout) that starts `offset` floats into its allocation."""
    n, D = x.shape
    buf = torch.zeros(D * env.pitch + offset, dtype=torch.float32, device=env.torch_device())
    t = buf[offset:].view(D, env.pitch)
    t[:, :n] = torch.from_numpy(np.ascontiguousarray(x.T)).to(t.device)
    return t


def _step(env, tr, N, torch, a, ncons, what, *, noise=None, reset_states=None, hostmask=None, want_obs=False,
          unpacked=False, action_offset=0):
    """One step_device call against one tracked oracle step: per-env outputs, state and episode words, then the statistics
    window of this step (counters, per-constraint counters, episode statistics, fp64 return sums); the window restarts."""
    orc, n = tr.orc, env.n
    out = {"reward": env.empty(), "flags": env.empty(dtype=torch.uint8), "viol_mask": env.empty(dtype=torch.uint8)}
    if want_obs:
        out["obs"], out["next_obs"] = env.empty(env.S), env.empty(env.S)
    if unpacked:
        out["terminated"], out["truncated"] = env.empty(dtype=torch.uint8), env.empty(dtype=torch.uint8)
    kw = {}
    if noise is not None:
        kw["noise"] = _soa(torch, env, noise)
    if reset_states is not None:
        kw["reset_states"] = _soa(torch, env, reset_states)
    if hostmask is not None:
        kw["hostmask"] = env.empty(dtype=torch.uint8)
        kw["hostmask"][:n] = torch.from_numpy(hostmask).to(kw["hostmask"].device)
    env.step_device(_soa(torch, env, a, action_offset), **kw, **out)
    o_ns, o_r, o_fl, o_vm = tr.step(a, noise=noise, reset_states=reset_states, hostmask=hostmask, want_next_obs=want_obs)
    torch.cuda.synchronize()
    got = {k: v[..., :n].cpu().numpy() for k, v in out.items()}
    assert_bits_equal(got["flags"], o_fl, f"{what}: flags")
    assert_bits_equal(got["viol_mask"], o_vm, f"{what}: violation mask")
    assert_bits_equal(got["reward"], o_r, f"{what}: reward")
    if want_obs:
        assert_bits_equal(got["next_obs"].T, o_ns, f"{what}: next_obs")
        assert_bits_equal(got["obs"].T, orc.state, f"{what}: obs")
    if unpacked:
        assert_bits_equal(got["terminated"], ((o_fl & 1) != 0).astype(np.uint8), f"{what}: terminated")
        assert_bits_equal(got["truncated"], ((o_fl & 2) != 0).astype(np.uint8), f"{what}: truncated")
    compare_state(env, orc, what)
    counters, sums = env.read_stats()
    compare_stats(N, counters, sums, tr, ncons, False, what, reward_sum=False)
    env.clear_stats()
    tr.clear()
    return counters


# ---------------------------------------------------------------------------------------------------------------------
# 1. dispatch witness
def test_step_dispatch_witness(mods, monkeypatch):
    """The single-step kernels the tests of this file (and the PowerGrid one of test_gpu_round2.py) are written for are the
    ones that run: recorded by name with torch.profiler."""
    ni, N, O, torch = mods
    from neorl_industrial.vector import make_constraint

    def names_of(kind, n, call, constraints=None, **envvars):
        for k, v in envvars.items():
            if v is None:
                monkeypatch.delenv(k, raising=False)
            else:
                monkeypatch.setenv(k, v)
        env = ni.NativeEnv(kind, n, device=0, seed=1, constraints=constraints)
        env.reset_device()
        got = kernel_names(torch, lambda: call(env))
        env.close()
        for k in envvars:
            monkeypatch.delenv(k, raising=False)
        return got

    def plain(e, offset=0, **kw):
        a = torch.zeros(e.A * e.pitch + offset, device=e.torch_device())[offset:].view(e.A, e.pitch)
        e.step_device(a, reward=e.empty(), flags=e.empty(dtype=torch.uint8), **kw)

    grid = names_of(N.ENV_POWER_GRID, GRID_N, plain, NIG_GRID_STEP=None)
    if not grid:
        pytest.skip("torch.profiler recorded no CUDA kernel in this process (no CUPTI activity records)")
    assert template_args(grid, "step_grid_kernel") == {("256", "128", "4")} and not template_args(grid, "step_kernel"), sorted(grid)
    g0 = names_of(N.ENV_POWER_GRID, GRID_N, plain, NIG_GRID_STEP="0")
    assert not template_args(g0, "step_grid_kernel") and template_args(g0, "step_kernel") == {("Grid", "1", "1", "true")}, sorted(g0)

    for name, env_t, vec in (("reactor", "Reactor", "2"), ("robot", "Robot", "1")):
        kind = KINDS[name]
        bound = make_constraint(N.CON_BOUND, si=0, lo=-1.0, hi=1.0, penalty=-5.0)
        pre = names_of(kind, PIPE_N[name], plain, constraints=_builtins(N, kind) + [bound])
        assert template_args(pre, "step_pipe_kernel") == {(env_t, vec, str(CONS_PREFIX))} and not template_args(pre, "step_kernel"), sorted(pre)
        gen = names_of(kind, PIPE_N[name], plain, constraints=_builtins(N, kind, (1, 0, 2)) + [bound])
        assert template_args(gen, "step_pipe_kernel") == {(env_t, vec, str(CONS_GENERIC))}, sorted(gen)

    R = N.ENV_CHEMICAL_REACTOR
    soa_obs = names_of(R, VEC2_N, lambda e: plain(e, obs=e.empty(e.S)))
    assert template_args(soa_obs, "step_kernel") == {("Reactor", "2", "1", "false")}, sorted(soa_obs)
    assert template_args(names_of(R, VEC2_N, plain), "step_pipe_kernel") == {("Reactor", "2", "1")}
    off8 = names_of(R, VEC2_N, lambda e: plain(e, 2))          # 8-byte aligned actions: no TMA pipeline, two envs per thread
    assert template_args(off8, "step_kernel") == {("Reactor", "2", "1", "false")} and not template_args(off8, "step_pipe_kernel"), sorted(off8)
    off4 = names_of(R, VEC2_N, lambda e: plain(e, 1))          # 4-byte aligned: one env per thread
    assert template_args(off4, "step_kernel") == {("Reactor", "1", "1", "true")}, sorted(off4)

    def aos_calls(e):              # nig_step_host on page-locked [n] arrays, and an AoS step_device call on the torch stream
        e.step_host(np.zeros((e.n, e.A), np.float32))
        e.step_device(torch.zeros((e.n, e.A), device=e.torch_device()), reward=e.empty(), flags=e.empty(dtype=torch.uint8),
                      action_layout=N.LAYOUT_AOS, aux_layout=N.LAYOUT_AOS)
    for vec in ("2", "4"):
        aos = names_of(R, 130, aos_calls, NIG_STEP_VEC=vec)
        assert {t[1] for t in template_args(aos, "step_kernel")} == {"1"}, (vec, sorted(aos))


# ---------------------------------------------------------------------------------------------------------------------
# 3. step_pipe_kernel with appended / re-ordered constraints
@pytest.mark.parametrize("auto_reset,pipe", [(True, "1"), (False, "1"), (True, "0")])
@pytest.mark.parametrize("cons", ["prefix", "generic"])
@pytest.mark.parametrize("name", ["reactor", "robot"])
def test_pipe_kernel_with_constraint_sets_vs_oracle(mods, monkeypatch, name, cons, auto_reset, pipe):
    """Plain step_device calls at populations above the pipe kernel's threshold with (prefix) the built-ins plus two
    SafetyWrapper bands -- step_pipe_kernel<Env, VEC, CONS_PREFIX> -- and (generic) re-ordered built-ins plus a bound plus
    host-mask descriptors that read 0 without a mask -- CONS_GENERIC. NIG_STEP_PIPE=0 runs the non-PLAIN step_kernel of
    the same set through the same oracle. The appended constraints must fire."""
    ni, N, O, torch = mods
    monkeypatch.setenv("NIG_STEP_PIPE", pipe)
    env, tr, ncons = _start(ni, N, O, name, PIPE_N[name], seed=71, env_id_offset=5, auto_reset=auto_reset, cons=cons)
    rng = np.random.default_rng(3)
    fired = np.zeros(ncons, np.int64)
    for t in range(4):
        c = _step(env, tr, N, torch, _actions(rng, env.n, env.A), ncons, f"{name} {cons} t={t}")
        fired += c[N.ST_CON0:N.ST_CON0 + ncons]
    assert (fired[3:4] > 0).all(), fired
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. step_kernel: vector width x constraint mode
_MATRIX = [("reactor", v, c) for v in (1, 2, 4) for c in ("prefix", "generic")] + \
          [(k, v, c) for k in ("grid", "robot") for v in (1, 2) for c in ("default", "prefix", "generic")]


@pytest.mark.parametrize("name,vec,cons", _MATRIX)
def test_step_kernel_vec_cons_matrix_vs_oracle(mods, monkeypatch, name, vec, cons):
    """Teacher-forced single steps (process noise, reset states, host masks) at 5,003 envs with SoA device arrays, obs /
    next_obs and the unpacked terminated / truncated outputs, for every vector width (NIG_STEP_VEC) and constraint mode."""
    ni, N, O, torch = mods
    monkeypatch.setenv("NIG_STEP_VEC", str(vec))
    env, tr, ncons = _start(ni, N, O, name, 5_003, seed=40 + vec, env_id_offset=11, cons=cons)
    rng = np.random.default_rng(vec)
    n = env.n
    for t in range(3):
        nz = rng.standard_normal((n, env.NZ)).astype(np.float32) if env.NZ else None
        rs = tr.orc.state[rng.permutation(n)].copy()
        hm = rng.integers(0, 4, n).astype(np.uint8) if cons == "generic" else None
        _step(env, tr, N, torch, _actions(rng, n, env.A), ncons, f"{name} VEC={vec} {cons} t={t}", noise=nz,
              reset_states=rs, hostmask=hm, want_obs=True, unpacked=True)
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. the reactor's two-env step kernel at its default dispatch
@pytest.mark.parametrize("variant", ["soa_obs", "noise", "actions_off8", "actions_off4"])
def test_reactor_vec2_default_dispatch_vs_oracle(mods, variant):
    """655,363 reactor envs (pitch >= 606,208): calls that are not plain take step_kernel<Reactor, 2>: SoA obs / next_obs
    outputs, teacher-forced noise, an action tensor 8 bytes past a 16-byte boundary (no TMA pipeline); one 4 bytes past
    it takes the one-env kernel, which has no alignment requirement."""
    ni, N, O, torch = mods
    env, tr, ncons = _start(ni, N, O, "reactor", VEC2_N, seed=5, env_id_offset=2)
    rng = np.random.default_rng(8)
    for t in range(3):
        nz = rng.standard_normal((env.n, env.NZ)).astype(np.float32) if variant == "noise" else None
        _step(env, tr, N, torch, _actions(rng, env.n, env.A), ncons, f"{variant} t={t}", noise=nz,
              want_obs=variant == "soa_obs", action_offset={"actions_off8": 2, "actions_off4": 1}.get(variant, 0))
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 6. persistent kernels in CUDA graphs
_GRAPH = {"grid_dedicated": ("grid", GRID_N), "reactor_pipe": ("reactor", PIPE_N["reactor"]),
          "robot_pipe": ("robot", PIPE_N["robot"]), "reactor_plain": ("reactor", 20_011)}


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("case", list(_GRAPH))
def test_persistent_step_kernels_graph_replay_vs_eager_and_oracle(mods, case, mode):
    """Three plain step_device calls captured in a CUDA graph (device tick mode 1, or mode 2 ending with commit_ticks) for
    the dedicated PowerGrid kernel (back to back under programmatic dependent launch), the reactor and robot pipe kernels
    and the PLAIN one-tile kernel, whose statistics go to per-warp shards folded on read: replays == eager calls == the
    oracle (state, episode words, counters, episode statistics), and the tick == the number of launches."""
    ni, N, O, torch = mods
    name, n = _GRAPH[case]
    kind = KINDS[name]
    envs = [ni.NativeEnv(kind, n, device=0, seed=31, env_id_offset=4) for _ in range(2)]
    graph_env, eager_env = envs
    orc = O.OracleEnv(kind, n, seed=31, env_id0=4, exp_mode=1, threads=O.max_threads())
    s0 = orc.reset()
    near = np.where(np.arange(n) % 5 == 0, graph_env.max_episode_steps - 4, 0).astype(np.int32)   # episodes end mid-run
    for e in envs:
        assert_bits_equal(e.reset_host(), s0, "reset draw")
        e.set_state_host(ep_step=near)
    orc.ep_step[:] = near
    tr = Track(orc, name)
    a_host = np.random.default_rng(kind).uniform(-1.1, 1.1, (n, graph_env.A)).astype(np.float32)
    acts = _soa(torch, graph_env, a_host)
    bufs = [(e.empty(), e.empty(dtype=torch.uint8), e.empty(dtype=torch.uint8)) for e in envs]

    def body(e, b):
        for _ in range(3):
            e.step_device(acts, reward=b[0], flags=b[1], viol_mask=b[2])

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
    for _ in range(4):
        g.replay()
        body(eager_env, bufs[1])
    for _ in range(15):
        o_r = tr.step(a_host, want_next_obs=False)[1]
    torch.cuda.synchronize()
    assert graph_env.tick == eager_env.tick == orc.tick == 15
    sg, stg, vg, dg = graph_env.get_state_host()
    se, ste, ve, de = eager_env.get_state_host()
    assert_bits_equal(sg, se, "state after graph replays vs eager")
    assert np.array_equal(stg, ste) and np.array_equal(vg, ve) and np.array_equal(dg, de)
    for e, b, what in ((graph_env, bufs[0], "graph"), (eager_env, bufs[1], "eager")):
        assert_bits_equal(b[0][:n].cpu().numpy(), o_r, f"{what}: last reward vs oracle")
        compare_state(e, orc, f"{what} vs oracle")
        counters, sums = e.read_stats()
        compare_stats(N, counters, sums, tr, 3, False, f"{what} statistics vs oracle", reward_sum=False)
    assert tr.len_sum > 0
    graph_env.use_device_tick(False)
    for e in envs:
        e.close()


# ---------------------------------------------------------------------------------------------------------------------
# 7. nig_step_host's terminated / truncated outputs
@pytest.mark.parametrize("zero_copy", ["1", "0"])
def test_step_host_terminated_truncated_vs_flags(mods, monkeypatch, zero_copy):
    """nig_step_host with terminated / truncated at 1,000 envs: pageable numpy arrays (the staged path), and page-locked
    ones with NIG_ZERO_COPY=0 (the staged path) or 1 (in place). Both arrays == the bits of flags == the oracle's, with
    episodes that truncate and episodes that terminate (critical temperature)."""
    ni, N, O, torch = mods
    monkeypatch.setenv("NIG_ZERO_COPY", zero_copy)
    n, S, A = 1_000, 12, 3
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=12)
    orc = O.OracleEnv(O.REACTOR, n, seed=12, exp_mode=1)
    s0 = env.reset_host().copy()
    assert_bits_equal(s0, orc.reset(), "reset draw")
    s0[:100, 0] = 356.0                                             # over the temperature limit: critical termination
    ep_step = np.where(np.arange(n) % 4 == 1, env.max_episode_steps - 1, 0).astype(np.int32)     # truncation
    env.set_state_host(s0, ep_step)
    orc.state[:] = s0
    orc.ep_step[:] = ep_step
    lib = N.lib()
    rng = np.random.default_rng(0)
    for pinned in (False, True):
        if pinned:
            alloc = lambda name, shape, dt: env.pinned("tt_" + name, shape, dt)
        else:
            alloc = lambda name, shape, dt: np.full(shape, 0xA5 if dt is np.uint8 else 0, dt)
        act, rew = alloc("act", (n, A), np.float32), alloc("rew", (n,), np.float32)
        fl, vm, term, trunc = (alloc(k, (n,), np.uint8) for k in ("fl", "vm", "term", "trunc"))
        act[:] = rng.uniform(-1, 1, (n, A)).astype(np.float32)
        term[:] = 0xA5; trunc[:] = 0xA5
        io = N.StepIO()
        io.actions, io.reward, io.flags, io.viol_mask = act.ctypes.data, rew.ctypes.data, fl.ctypes.data, vm.ctypes.data
        io.terminated, io.truncated = term.ctypes.data, trunc.ctypes.data
        io.action_layout, io.aux_layout = N.LAYOUT_AOS, N.LAYOUT_AOS
        N.check(lib.nig_step_host(env._h, C.byref(io)))
        _, o_r, o_fl, o_vm = orc.step(act.copy(), want_next_obs=False)
        what = f"pinned={pinned} zero_copy={zero_copy}"
        assert_bits_equal(fl, o_fl, f"{what}: flags")
        assert_bits_equal(rew, o_r, f"{what}: reward")
        assert_bits_equal(term, ((fl & 1) != 0).astype(np.uint8), f"{what}: terminated")
        assert_bits_equal(trunc, ((fl & 2) != 0).astype(np.uint8), f"{what}: truncated")
        if not pinned:
            assert term.sum() >= 100 and trunc.sum() >= 200, what
    compare_state(env, orc, "after the host steps")
    env.close()
