"""The kernels at the limits of their counters: the episode word (16-bit step at max_episode_steps = 65,535, 15-bit
saturating violation count), the uint32 RNG tick across its wrap (single launches, sliced and graph-replayed calls, the
host-buffer call, the device-tick modes, a checkpoint), the reset epoch's period of 2^24, the 32-bit global env ids, and
the statistics of one fused launch at NIG_MAX_LAUNCH_STEPS. Every kernel family is compared with the CPU oracle
(spec-exp mode) bit for bit, the fp64 statistics to the tolerances of tests/test_gpu_parity.py; the counts at the launch
bound are known exactly. A dispatch witness records kernel names so that no case loses its kernel silently."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from util import KINDS, Track, assert_bits_equal, compare_stats, kernel_names, set_population, start_pair, template_args

pytestmark = pytest.mark.gpu

KMAX = 1 << 20                      # NIG_MAX_LAUNCH_STEPS
WRAP0 = (1 << 32) - 13              # a tick 13 steps before the uint32 wrap
EP_CAP = 65_535                     # the largest max_episode_steps: the whole 16-bit step field
VIOL_SAT = 32_767                   # the episode word's violation count saturates here
CONS_GENERIC, CONS_DEFAULT, CONS_BOUNDS2 = 0, 1, 4      # nig_kernels.cuh

# every kernel family, at the size or switch that selects it on a B200 (148 SMs; see test_dispatch_witness):
# (operation, env, envs, environment variables)
FAMILIES = {
    "rollout_reactor_warp": ("rollout", "reactor", 4_099, {}),           # fast loop, one-warp CTAs (<= 16,384 envs)
    "rollout_reactor_cta128": ("rollout", "reactor", 20_011, {}),        # fast loop, 128-thread CTAs
    "rollout_reactor_bands": ("rollout", "reactor", 4_099, {}),          # fast loop with two wrapper bands (FastBounds)
    "rollout_reactor_pair": ("rollout", "reactor", 131_072 + 99, {}),    # rollout_reactor_pair_kernel
    "rollout_grid": ("rollout", "grid", 4_133, {}),                      # rollout_grid_kernel
    "rollout_grid_generic": ("rollout", "grid", 4_133, {"NIG_GRID_FAST": "0"}),
    "rollout_robot": ("rollout", "robot", 4_133, {}),
    "rollout_mlp": ("rollout", "reactor", 4_133, {}),                    # rollout_mlp_kernel
    "step_plain": ("step", "reactor", 20_011, {}),                       # step_kernel<..., PLAIN>
    "step_vec1": ("step", "reactor", 5_003, {"NIG_STEP_VEC": "1"}),
    "step_vec2": ("step", "reactor", 5_003, {"NIG_STEP_VEC": "2"}),
    "step_vec4": ("step", "reactor", 5_003, {"NIG_STEP_VEC": "4"}),
    "step_aos": ("step", "reactor", 5_003, {"NIG_STEP_VEC": "4"}),       # AoS layouts always take VEC = 1
    "step_pipe_reactor": ("step", "reactor", 151_553, {}),               # step_pipe_kernel above 151,552 reactor envs
    "step_pipe_robot": ("step", "robot", 75_777, {}),                    # ... and above 75,776 robot envs
    "step_grid": ("step", "grid", 227_073, {}),                          # step_grid_kernel from 227,073 envs
}


@pytest.fixture(scope="module")
def mods():
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    from oracle import oracle as O
    return ni, N, O, torch


def _bands(N):
    """The reactor's built-ins plus two empty SafetyWrapper bands (lo > hi: violated on every step) on T and P: the
    straight-line CONS_BOUNDS2 loop."""
    from neorl_industrial.vector import make_constraint
    spec = N.env_spec(N.ENV_CHEMICAL_REACTOR)
    return [make_constraint(N.CON_BUILTIN, cid=k, penalty=spec.constraints[k].penalty, critical=bool(spec.constraints[k].critical))
            for k in range(3)] + [make_constraint(N.CON_BOUND, si=si, lo=1.0, hi=0.0, penalty=-3.0) for si in (0, 1)]


def _empty8(N):
    """Eight empty bounds (lo > hi) and no built-in: every env violates all eight on every step (CONS_GENERIC)."""
    from neorl_industrial.vector import make_constraint
    return [make_constraint(N.CON_BOUND, si=k, lo=1.0, hi=0.0, penalty=-0.25) for k in range(8)]


def _mlp(ni, S, A):
    """A small one-hidden-layer network with identity output (actions beyond +-1 exercise the env's clip)."""
    rng = np.random.default_rng(5)
    return ni.MLPPolicy([rng.normal(0, 0.02, (64, S)).astype(np.float32), rng.normal(0, 0.3, (A, 64)).astype(np.float32)],
                        output_activation="identity")


def _soa(torch, env, x):
    t = torch.zeros((x.shape[1], env.pitch), dtype=torch.float32, device=env.torch_device())
    t[:, :x.shape[0]] = torch.from_numpy(np.ascontiguousarray(x.T)).to(t.device)
    return t


def _call(N, torch, fam, env, K, a=None, out=None):
    """The family's operation: one fused K-step launch, or one single step with actions a [n, A] (zeros when None)."""
    op = FAMILIES[fam][0]
    if op == "rollout":
        policy = N.POLICY_MLP if fam == "rollout_mlp" else N.POLICY_UNIFORM
        env.rollout_device(K, policy, **(out or {}))
        return
    a = np.zeros((env.n, env.A), np.float32) if a is None else a
    out = dict(out or {})
    if fam == "step_aos":
        env.step_device(torch.from_numpy(a).to(env.torch_device()), action_layout=N.LAYOUT_AOS, aux_layout=N.LAYOUT_AOS, **out)
        return
    if fam.startswith("step_vec"):           # an observation output: not the plain flavour
        out.setdefault("obs", env.empty(env.S))
    env.step_device(_soa(torch, env, a), **out)


def _make(mods, monkeypatch, fam, *, seed, max_steps=None, auto_reset=True, constraints=None, env_id_offset=7):
    ni, N, O, torch = mods
    _, name, n, envvars = FAMILIES[fam]
    for k, v in envvars.items():
        monkeypatch.setenv(k, v)
    if constraints is None and fam == "rollout_reactor_bands":
        constraints = _bands(N)
    env, orc = start_pair(ni, O, KINDS[name], n, seed=seed, env_id_offset=env_id_offset, max_episode_steps=max_steps,
                          auto_reset=auto_reset, constraints=constraints, threads=O.max_threads())
    if fam == "rollout_mlp":
        env.set_mlp_policy(_mlp(ni, env.S, env.A))
    return env, orc, Track(orc, name), 3 if constraints is None else len(constraints)


def compare_state_saturated(env, orc, what):
    """get_state == the oracle's, with the episode violation count saturated at 32,767 (the oracle's count does not)."""
    st, ep_step, ep_viol, done = env.get_state_host()
    assert_bits_equal(st, orc.state, f"{what}: state")
    assert_bits_equal(ep_step, orc.ep_step, f"{what}: episode step")
    assert_bits_equal(ep_viol, np.minimum(orc.ep_viol, VIOL_SAT), f"{what}: episode violations")
    assert_bits_equal(done, orc.done_latch.astype(bool), f"{what}: done latch")


def _run(mods, fam, env, orc, tr, ncons, chunks, what, seed=0):
    """The family's launches against the tracked oracle. Rollouts: one K-step launch per chunk; single steps: K steps per
    chunk. After every launch: per-env outputs, state and the three get_state fields, and the statistics window (counters,
    per-constraint counters, episode count / length sum / length square sum, fp64 sums), which then restarts."""
    ni, N, O, torch = mods
    n, op = orc.n, FAMILIES[fam][0]
    rng = np.random.default_rng(seed)
    if op == "rollout":
        policy = (lambda: env.selftest_mlp(orc.state)) if fam == "rollout_mlp" else (lambda: O.policy_actions(orc, O.POLICY_UNIFORM))
        rsum, vcnt, dcnt = env.empty(), env.empty(dtype=torch.int32), env.empty(dtype=torch.int32)
    for K in chunks:
        for t in range(1 if op == "rollout" else K):
            w = f"{what}, {fam}: launch of {K} steps" if op == "rollout" else f"{what}, {fam}: step {t} of {K}"
            if op == "rollout":
                _call(N, torch, fam, env, K, out={"reward_sum": rsum, "viol_count": vcnt, "done_count": dcnt})
                o_rs, o_v, o_d = tr.launch(K, policy)
                torch.cuda.synchronize()
                assert_bits_equal(rsum[:n].cpu().numpy(), o_rs, f"{w}: per-env reward sum")
                assert_bits_equal(vcnt[:n].cpu().numpy().astype(np.int64), o_v, f"{w}: per-env violation count")
                assert_bits_equal(dcnt[:n].cpu().numpy().astype(np.int64), o_d, f"{w}: per-env done count")
            else:
                a = rng.uniform(-1.1, 1.1, (n, env.A)).astype(np.float32)
                out = {"reward": env.empty(), "flags": env.empty(dtype=torch.uint8), "viol_mask": env.empty(dtype=torch.uint8)}
                _call(N, torch, fam, env, 1, a, out)
                _, o_r, o_fl, o_vm = tr.step(a, want_next_obs=False)
                torch.cuda.synchronize()
                assert_bits_equal(out["flags"][:n].cpu().numpy(), o_fl, f"{w}: flags")
                assert_bits_equal(out["viol_mask"][:n].cpu().numpy(), o_vm, f"{w}: violation mask")
                assert_bits_equal(out["reward"][:n].cpu().numpy(), o_r, f"{w}: reward")
            compare_state_saturated(env, orc, w)
            counters, sums = env.read_stats()
            compare_stats(N, counters, sums, tr, ncons, False, w, reward_sum=op == "rollout")
            env.clear_stats()
            tr.clear()
    assert env.tick == orc.tick % (1 << 32), (env.tick, orc.tick)


# ---------------------------------------------------------------------------------------------------------------------
# 1. dispatch witness
def _dispatch_names():
    """Prints, as JSON, the kernel names torch.profiler records for one call of every family (and of the saturation and
    launch-bound constraint sets)."""
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    out = {}
    cases = [(fam, None) for fam in FAMILIES] + [("rollout_reactor_warp", "empty8"), ("rollout_reactor_cta128", "empty8"),
                                                 ("rollout_grid", "empty8"), ("rollout_robot", "empty8")]
    for fam, cons in cases:
        _, name, n, envvars = FAMILIES[fam]
        os.environ.update(envvars)
        cs = _empty8(N) if cons else (_bands(N) if fam == "rollout_reactor_bands" else None)
        env = ni.NativeEnv(KINDS[name], n, device=0, seed=1, constraints=cs)
        env.reset_device()
        if fam == "rollout_mlp":
            env.set_mlp_policy(_mlp(ni, env.S, env.A))
        out[f"{fam} {cons}"] = sorted(kernel_names(torch, lambda: _call(N, torch, fam, env, 8)))
        env.close()
        for k in envvars:
            del os.environ[k]
    print(json.dumps(out))


def test_dispatch_witness():
    """Every family runs the kernel it is named for. Recorded in a child process, like test_gpu_dataset_flavours.py's
    witness, so that the profiler session does not disturb the witnesses of the other files."""
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    code = (f"import sys; sys.path[:0] = {[root, os.path.join(root, 'neorl-industrial-gym_b200'), here]!r}; "
            "import test_gpu_limits as t; t._dispatch_names()")
    flags = ["-s"] if sys.flags.no_user_site else []
    run = subprocess.run([sys.executable, *flags, "-c", code], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr[-8000:]
    got = json.loads(run.stdout.strip().splitlines()[-1])
    if not any(got.values()):
        pytest.skip("torch.profiler recorded no CUDA kernel in the child process (no CUPTI activity records)")
    roll = lambda k: template_args(got[k], "rollout_kernel")
    step = lambda k: template_args(got[k], "step_kernel")
    D, U = str(CONS_DEFAULT), "1"                      # CONS_DEFAULT, NIG_POLICY_UNIFORM
    assert roll("rollout_reactor_warp None") == {("Reactor", D, U, "false", "false", "false")}, got
    assert roll("rollout_reactor_cta128 None") == {("Reactor", D, U, "false", "false", "false")}, got
    assert roll("rollout_reactor_bands None") == {("Reactor", str(CONS_BOUNDS2), U, "false", "false", "false")}, got
    assert any("rollout_reactor_pair_kernel" in x for x in got["rollout_reactor_pair None"]), got
    assert not roll("rollout_reactor_pair None"), got
    assert any("rollout_grid_kernel" in x for x in got["rollout_grid None"]) and not roll("rollout_grid None"), got
    assert roll("rollout_grid_generic None") == {("Grid", D, U, "false", "false", "false")}, got
    assert roll("rollout_robot None") == {("Robot", D, U, "false", "false", "false")}, got
    assert any("rollout_mlp_kernel" in x for x in got["rollout_mlp None"]), got
    for fam, env_t in (("rollout_reactor_warp", "Reactor"), ("rollout_reactor_cta128", "Reactor"), ("rollout_grid", "Grid"),
                       ("rollout_robot", "Robot")):
        assert roll(f"{fam} empty8") == {(env_t, str(CONS_GENERIC), U, "false", "false", "false")}, got
    assert step("step_plain None") == {("Reactor", "1", D, "true")}, got
    for v in ("1", "2", "4"):
        assert step(f"step_vec{v} None") == {("Reactor", v, D, "false")}, got
    assert step("step_aos None") == {("Reactor", "1", D, "false")}, got
    assert template_args(got["step_pipe_reactor None"], "step_pipe_kernel") == {("Reactor", "2", D)}, got
    assert template_args(got["step_pipe_robot None"], "step_pipe_kernel") == {("Robot", "1", D)}, got
    assert template_args(got["step_grid None"], "step_grid_kernel") and not step("step_grid None"), got


# ---------------------------------------------------------------------------------------------------------------------
# 2. the episode step at 65,535
def _near_cap(n, cap):
    """ep_step = cap - j: four lanes of every 32 share each of eight truncation steps 1, 4, .., 22 of a 24-step launch,
    every fifth warp truncates 24 steps later (in the second launch)."""
    i = np.arange(n)
    j = 1 + 3 * (i % 8) + 24 * ((i // 32) % 5 == 4)
    return (cap - j).astype(np.int32)


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("fam", list(FAMILIES))
def test_episode_step_at_65535_vs_oracle(mods, monkeypatch, fam, auto_reset):
    """max_episode_steps = 65,535 with episodes 1 to 46 steps before the cap: truncations at different steps of one launch,
    a whole warp's episodes of ~65,535 steps in one launch (a length-square sum near 2^37), done latches at step 65,535
    without auto-reset. Two 24-step launches (48 single steps) == the oracle after every launch."""
    env, orc, tr, ncons = _make(mods, monkeypatch, fam, seed=17, max_steps=EP_CAP, auto_reset=auto_reset)
    set_population(env, orc, orc.state.copy(), _near_cap(orc.n, EP_CAP))
    _run(mods, fam, env, orc, tr, ncons, (24, 24), "ep_step near 65,535")
    assert (orc.ep_step == EP_CAP).any() == (not auto_reset)
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. violation count saturation
@pytest.mark.parametrize("case", ["reactor_bands", "reactor_empty8", "grid_empty8", "robot_empty8"])
def test_violation_count_saturates_vs_oracle(mods, monkeypatch, case):
    """Imported episode violation counts 32,767 - j under two constraint sets that violate on every step: the reactor's two
    empty bands (the CONS_BOUNDS2 fast loop: + 2 per step) and eight empty bounds (CONS_GENERIC: + 8 per step) for every env.
    get_state's count == min(oracle, 32,767); per-env viol_count, statistics, the done latch and everything else == the
    oracle's exact counts."""
    ni, N, O, torch = mods
    name, cons = case.split("_")
    fam = {"reactor": "rollout_reactor_warp", "grid": "rollout_grid", "robot": "rollout_robot"}[name]
    cs = _bands(N) if cons == "bands" else _empty8(N)
    env, orc, tr, ncons = _make(mods, monkeypatch, fam, seed=23, max_steps=40, constraints=cs)
    n = orc.n
    ep_step = (np.arange(n) % 37).astype(np.int32)
    ep_viol = (VIOL_SAT - np.arange(n) % 64).astype(np.int32)
    set_population(env, orc, orc.state.copy(), ep_step, ep_viol=ep_viol)
    _run(mods, fam, env, orc, tr, ncons, (24, 5), f"saturation {case}")
    assert (orc.ep_viol > VIOL_SAT).any()
    env.close()


def test_single_env_host_counter_vs_saturated_device_field(mods):
    """One RobotAssembly-v0 env through ni.make with eight empty bounds and max_episode_steps = 65,535, zero actions for
    4,100 steps (the oracle shows the episode running on): 32,800 violations. The single-env API's host counter keeps
    them all (like the reference's int), get_state's device field saturates at 32,767."""
    ni, N, O, torch = mods
    env = ni.make("RobotAssembly-v0", seed=3, env_id_offset=1, max_episode_steps=EP_CAP)
    for c in list(env.safety_constraints):
        env.remove_safety_constraint(c.name)
    for k in range(8):
        env.add_safety_constraint(ni.BoundConstraint(f"empty{k}", k, 1.0, 0.0, penalty=-0.25))
    orc = O.OracleEnv(O.ROBOT, 1, env_id0=1, seed=3, exp_mode=1, auto_reset=False, builtin=False, max_episode_steps=EP_CAP,
                      extra_cons=[O.Con(N.CON_BOUND, 0, k, -1, 0.0, 1.0, 0.0, -0.25, 0) for k in range(8)])
    obs, _ = env.reset()
    assert_bits_equal(obs[None], orc.reset(), "reset draw")
    a = np.zeros(env.action_dim, np.float32)
    for t in range(4_100):
        obs, r, term, trunc, info = env.step(a)
        _, o_r, o_fl, _ = orc.step(a[None], want_next_obs=False)
        assert not (term or trunc) and o_fl[0] & 3 == 0, t
    assert_bits_equal(obs[None], orc.state, "state after 4,100 steps")
    assert env.violation_count == info["violations"] == int(orc.ep_viol[0]) == 8 * 4_100
    assert env.current_step == 4_100
    ckpt = env.get_state()
    assert int(ckpt["ep_viol"][0]) == VIOL_SAT and int(ckpt["ep_step"][0]) == 4_100
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. the tick across its wrap
def _ending(n, cap):
    """Episodes ending on every step of the first 40 (their resets draw at ticks on both sides of the wrap)."""
    return (cap - 1 - np.arange(n) % 40).astype(np.int32)


@pytest.mark.parametrize("fam", list(FAMILIES))
def test_tick_wrap_vs_oracle(mods, monkeypatch, fam):
    """Tick 2^32 - 13 on both sides, then a 24-step launch (24 single steps) across the wrap and an 8-step one after it,
    with episodes ending and auto-resetting on every step."""
    env, orc, tr, ncons = _make(mods, monkeypatch, fam, seed=29)
    set_population(env, orc, orc.state.copy(), _ending(orc.n, env.max_episode_steps))
    env.set_tick(WRAP0)
    orc.tick = WRAP0
    assert env.tick == WRAP0
    _run(mods, fam, env, orc, tr, ncons, (24, 8), "across the tick wrap")
    assert env.tick == 19
    env.close()


def _chunked(tr, T, K, policy):
    """The oracle side of one T-step call made of ceil(T / K) launches: per-env fp32 sums added launch by launch."""
    total, o_v, o_d = None, 0, 0
    for c0 in range(0, T, K):
        part, v, d = tr.launch(min(K, T - c0), policy)
        total = part if total is None else (total + part).astype(np.float32)
        o_v, o_d = o_v + v, o_d + d
    return total, o_v, o_d


@pytest.mark.parametrize("slices,graph", [(1, "1"), (8, "1"), (8, "0")])
def test_rollout_steps_across_tick_wrap_vs_oracle(mods, monkeypatch, slices, graph):
    """nig_rollout_steps at 69,635 reactor envs, three calls of 20 steps in 8-step launches from tick 2^32 - 30: the second
    call crosses the wrap. One slice (the plain launch sequence), or eight (the first call enqueued launch by launch, the
    second captured and the third replayed as a CUDA graph; NIG_STEPS_GRAPH=0: never)."""
    ni, N, O, torch = mods
    monkeypatch.setenv("NIG_HOST_SLICES", str(slices))
    monkeypatch.setenv("NIG_STEPS_GRAPH", graph)
    n, T, K = 69_635, 20, 8
    env, orc = start_pair(ni, O, O.REACTOR, n, seed=31, env_id_offset=3, max_episode_steps=60, threads=O.max_threads())
    set_population(env, orc, orc.state.copy(), _ending(n, 60))
    env.set_tick((1 << 32) - 30)
    orc.tick = (1 << 32) - 30
    tr = Track(orc, "reactor")
    policy = lambda: O.policy_actions(orc, O.POLICY_UNIFORM)
    rsum, vcnt, dcnt = env.empty(), env.empty(dtype=torch.int32), env.empty(dtype=torch.int32)
    for call in range(3):
        env.rollout_steps_device(T, K, N.POLICY_UNIFORM, reward_sum=rsum, viol_count=vcnt, done_count=dcnt)
        total, o_v, o_d = _chunked(tr, T, K, policy)
        torch.cuda.synchronize()
        w = f"call {call}, {slices} slices, graph={graph}"
        assert_bits_equal(rsum[:n].cpu().numpy(), total, f"{w}: per-env reward sum")
        assert np.array_equal(vcnt[:n].cpu().numpy(), o_v) and np.array_equal(dcnt[:n].cpu().numpy(), o_d), w
        compare_state_saturated(env, orc, w)
        counters, sums = env.read_stats()
        compare_stats(N, counters, sums, tr, 3, False, w)
        env.clear_stats()
        tr.clear()
        assert env.tick == orc.tick % (1 << 32), w
    env.close()


@pytest.mark.parametrize("direct", [True, False])
def test_rollout_host_across_tick_wrap_vs_oracle(mods, monkeypatch, direct):
    """nig_rollout_host at 69,635 reactor envs, sliced, through the direct path (the slices' kernels read / write the
    page-locked arrays) and the staged one, each captured as one graph whose launches take the tick as an offset from a
    base word: two calls of 20 steps in 8-step launches from tick 2^32 - 25, the second (a replay) across the wrap."""
    ni, N, O, torch = mods
    monkeypatch.setenv("NIG_HOST_DIRECT", "3" if direct else "0")
    monkeypatch.setenv("NIG_HOST_DIRECT_MAX_MB", "1e9")
    n, T, K = 69_635, 20, 8
    env, orc = start_pair(ni, O, O.REACTOR, n, seed=37, env_id_offset=11, max_episode_steps=60, threads=O.max_threads())
    set_population(env, orc, orc.state.copy(), _ending(n, 60))
    env.set_tick((1 << 32) - 25)
    orc.tick = (1 << 32) - 25
    tr = Track(orc, "reactor")
    for call in range(2):
        out = env.rollout_host(T, N.POLICY_UNIFORM, steps_per_launch=K)
        total, o_v, o_d = _chunked(tr, T, K, lambda: O.policy_actions(orc, O.POLICY_UNIFORM))
        w = f"host call {call}, direct={direct}"
        assert_bits_equal(out["obs"], orc.state, f"{w}: final observations")
        assert_bits_equal(out["reward_sum"], total, f"{w}: per-env reward sum")
        assert np.array_equal(out["violations"], o_v) and np.array_equal(out["episodes"], o_d), w
        compare_state_saturated(env, orc, w)
        compare_stats(N, out["counters"], out["sums"], tr, 3, False, w)
        assert env.tick == orc.tick % (1 << 32), w
    env.close()


@pytest.mark.parametrize("mode", [1, 2])
def test_device_tick_graph_across_wrap_vs_eager_and_oracle(mods, mode):
    """test_gpu_graph.py's captured sequence (single steps + a 16-step fused rollout, 19 ticks) from tick 2^32 - 50 with the
    device-resident tick (mode 1: advanced by every launch; mode 2: base + per-launch offsets, committed at the end): five
    runs cross the wrap. Replays == eager stepping (mode 0) == the oracle, and nig_get_tick agrees in every mode."""
    ni, N, O, torch = mods
    n, t0 = 4_099, (1 << 32) - 50
    envs = [ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=41, env_id_offset=2, max_episode_steps=30) for _ in range(2)]
    graph_env, eager_env = envs
    orc = O.OracleEnv(O.REACTOR, n, seed=41, env_id0=2, exp_mode=1, max_episode_steps=30)
    s0 = orc.reset()
    for e in envs:
        assert_bits_equal(e.reset_host(), s0, "reset draw")
        e.set_tick(t0)
    orc.tick = t0
    acts = torch.rand((graph_env.A, graph_env.pitch), device=graph_env.torch_device()) * 2 - 1
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
    assert graph_env.tick == t0
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
    for _ in range(5):
        o_r = oracle_body()
    torch.cuda.synchronize()
    assert graph_env.tick == eager_env.tick == orc.tick % (1 << 32) == t0 + 5 * 19 - (1 << 32)
    sg, stg, vg, dg = graph_env.get_state_host()
    assert_bits_equal(sg, orc.state, "graph replays vs oracle: state")
    assert np.array_equal(stg, orc.ep_step) and np.array_equal(vg, orc.ep_viol)
    compare_state_saturated(eager_env, orc, "eager vs oracle")
    for b in bufs:
        assert_bits_equal(b[0][:n].cpu().numpy(), o_r, "last reward vs oracle")
    cg, _ = graph_env.read_stats()
    ce, _ = eager_env.read_stats()
    assert cg[:8].tolist() == ce[:8].tolist() and ce[:6].tolist() == orc.stats[:6].tolist()
    graph_env.use_device_tick(False)
    assert graph_env.tick == orc.tick % (1 << 32)
    for e in envs:
        e.close()


def test_checkpoint_round_trip_across_wrap(mods):
    """IndustrialEnv.get_state at tick 2^32 - 13, a 24-step launch across the wrap; set_state(checkpoint) and the same
    launch again give the same bits, and both == the oracle."""
    ni, N, O, torch = mods
    n = 4_099
    env = ni.ChemicalReactorEnv(num_envs=n, seed=43, env_id_offset=6, max_episode_steps=50)
    orc = O.OracleEnv(O.REACTOR, n, seed=43, env_id0=6, exp_mode=1, max_episode_steps=50)
    obs, _ = env.reset()
    assert_bits_equal(obs, orc.reset(), "reset draw")
    env.native.set_tick(WRAP0)
    orc.tick = WRAP0
    env.native.rollout_device(5, N.POLICY_UNIFORM)
    tr = Track(orc, "reactor")
    tr.launch(5, lambda: O.policy_actions(orc, O.POLICY_UNIFORM))
    ckpt = env.get_state()
    assert ckpt["tick"] == WRAP0 + 5
    runs = []
    for _ in range(2):
        env.native.rollout_device(24, N.POLICY_UNIFORM)
        runs.append(env.native.get_state_host() + (env.native.tick,))
        env.set_state(ckpt)
    tr.launch(24, lambda: O.policy_actions(orc, O.POLICY_UNIFORM))
    for k, what in enumerate(("state", "episode step", "episode violations", "done")):
        assert_bits_equal(runs[1][k], runs[0][k], f"restored run: {what}")
    assert runs[0][4] == runs[1][4] == orc.tick % (1 << 32) == 16
    assert_bits_equal(runs[0][0], orc.state, "state vs oracle")
    assert np.array_equal(runs[0][1], orc.ep_step)
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. the reset epoch and the global env ids
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_reset_epoch_period(mods, name):
    """Explicit resets draw with the counter word (epoch << 8) | j: the reset at epoch 2^24 == the oracle's, and == the
    draw at epoch 0 at the same tick (a period of 2^24 explicit resets, part of the RNG spec)."""
    ni, N, O, torch = mods
    kind, n, tick = KINDS[name], 1_000, 123_457
    env = ni.NativeEnv(kind, n, device=0, seed=47, env_id_offset=8)
    env.set_tick(tick, (1 << 24) - 1)
    got = env.reset_host().copy()
    assert env.epoch == 1 << 24
    draws = []
    for epoch in ((1 << 24) - 1, -1):             # OracleEnv.reset draws with epoch + 1
        orc = O.OracleEnv(kind, n, seed=47, env_id0=8, exp_mode=1)
        orc.tick, orc.epoch = tick, epoch
        draws.append(orc.reset())
    assert_bits_equal(got, draws[0], "reset at epoch 2^24 vs oracle")
    assert_bits_equal(got, draws[1], "reset at epoch 2^24 vs epoch 0")
    other = O.OracleEnv(kind, n, seed=47, env_id0=8, exp_mode=1)
    other.tick = tick
    assert not np.array_equal(got, other.reset()), "epoch 1 must draw differently"
    env.close()


def test_last_env_ids_vs_oracle(mods):
    """A handle whose envs are the last 100 global ids (env_id_offset = 2^32 - 100): reset, a rollout, single steps and a
    dataset == the oracle's; one id more is rejected, at creation and by the dataset calls."""
    ni, N, O, torch = mods
    off = (1 << 32) - 100
    env, orc = start_pair(ni, O, O.REACTOR, 100, seed=53, env_id_offset=off, max_episode_steps=20)
    tr = Track(orc, "reactor")
    _run(mods, "rollout_reactor_warp", env, orc, tr, 3, (30,), "last ids")
    a = np.random.default_rng(0).uniform(-1, 1, (100, 3)).astype(np.float32)
    obs, _, r, fl, vm = env.step_host(a)
    _, o_r, o_fl, o_vm = orc.step(a, want_next_obs=False)
    assert_bits_equal(obs, orc.state, "step state")
    assert_bits_equal(r, o_r, "step reward")
    assert_bits_equal(fl, o_fl, "step flags")
    pp = N.PolicyParams()
    assert env.dataset_size(100, 30, N.POLICY_UNIFORM, pp) > 0
    with pytest.raises(ValueError, match="2\\^32"):
        env.dataset_size(101, 30, N.POLICY_UNIFORM, pp)
    env.close()
    for bad in (off + 1, -1):
        with pytest.raises(ValueError, match="2\\^32"):
            ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, 100, device=0, env_id_offset=bad)


def test_imports_outside_the_word_are_rejected_or_clamped(mods):
    """nig_set_state_host (and the Python setters above it) rejects an episode step outside [0, 65535] and a negative
    violation count, importing nothing; a count above 32,767 saturates. nig_set_state clamps device arrays into range."""
    ni, N, O, torch = mods
    env = ni.ChemicalReactorEnv(num_envs=256, seed=59)
    env.reset()
    before = env.native.get_state_host()
    for kw in ({"ep_step": np.full(256, 65_536)}, {"ep_step": np.full(256, -1)}, {"ep_viol": np.full(256, -1)}):
        with pytest.raises(ValueError):
            env.native.set_state_host(**kw)
    with pytest.raises(ValueError):
        env.current_step = 65_536
    with pytest.raises(ValueError):
        env.violation_count = -5
    ckpt = env.get_state()
    ckpt["ep_step"] = ckpt["ep_step"].copy()
    ckpt["ep_step"][7] = 70_000
    with pytest.raises(ValueError):
        env.set_state(ckpt)
    after = env.native.get_state_host()
    for x, y in zip(before, after):
        assert np.array_equal(x, y), "a rejected import changed the state"
    env.current_step = 65_535
    env.violation_count = 40_000
    _, st, vi, _ = env.native.get_state_host()
    assert (st == 65_535).all() and (vi == VIOL_SAT).all()
    dev = env.native.torch_device()
    steps = torch.tensor([70_000, -3, 65_535, 12] * 64, dtype=torch.int32, device=dev)
    viols = torch.tensor([-1, 40_000, 5, VIOL_SAT] * 64, dtype=torch.int32, device=dev)
    env.native.set_state_device(ep_step=steps, ep_viol=viols)
    torch.cuda.synchronize()
    _, st, vi, dn = env.native.get_state_host()
    assert st.tolist() == [65_535, 0, 65_535, 12] * 64 and vi.tolist() == [0, VIOL_SAT, 5, VIOL_SAT] * 64
    assert not dn.any()
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 6. statistics at the launch bound
@pytest.mark.parametrize("n", [148 * 128 + 77, 4_099], ids=["cta128_ragged", "one_warp"])
def test_statistics_at_launch_bound(mods, monkeypatch, n):
    """Eight empty bounds (8 violations per env-step) with NIG_POLICY_ZERO at 148 x 128 + 77 reactor envs (128-thread CTAs,
    the last one ragged) and 4,099 (one-warp CTAs). First 64 steps == the oracle (the set behaves as specified); then one
    launch of NIG_MAX_LAUNCH_STEPS steps, and a host call of 2^22 + 3 steps with steps_per_launch = 0 (capped to launches
    of NIG_MAX_LAUNCH_STEPS) in one slice: steps, violations, per-constraint counts, per-env violation counts and episodes
    are exact. (In one launch, the 128-thread CTAs' shared violation slots would wrap.) One step more per launch is
    rejected."""
    ni, N, O, torch = mods
    monkeypatch.setenv("NIG_HOST_SLICES", "1")
    cs = _empty8(N)
    env, orc = start_pair(ni, O, O.REACTOR, n, seed=61, constraints=cs, threads=O.max_threads())
    tr = Track(orc, "reactor")
    rsum, vcnt, dcnt = env.empty(), env.empty(dtype=torch.int32), env.empty(dtype=torch.int32)
    env.rollout_device(64, N.POLICY_ZERO, reward_sum=rsum, viol_count=vcnt, done_count=dcnt)
    o_rs, o_v, o_d = tr.launch(64, lambda: O.policy_actions(orc, O.POLICY_ZERO))
    torch.cuda.synchronize()
    assert_bits_equal(rsum[:n].cpu().numpy(), o_rs, "64 steps: per-env reward sum")
    assert np.array_equal(vcnt[:n].cpu().numpy(), o_v) and np.array_equal(dcnt[:n].cpu().numpy(), o_d)
    compare_state_saturated(env, orc, "64 steps")
    counters, sums = env.read_stats()
    compare_stats(N, counters, sums, tr, 8, False, "64 steps")
    assert (o_v == 8 * 64).all()

    def exact(counters, viol, done, K, what):
        nk = n * K
        assert int(counters[N.ST_STEPS]) == nk, (what, counters[:8])
        assert int(counters[N.ST_VIOLATIONS]) == 8 * nk, (what, counters[:8])
        assert counters[N.ST_CON0:N.ST_CON0 + 8].tolist() == [nk] * 8, (what, counters[8:16])
        assert (viol == 8 * K).all() and int(viol.astype(np.int64).sum()) == 8 * nk, what
        assert int(done.astype(np.int64).sum()) == int(counters[N.ST_EPISODES]) > 0, what

    env.clear_stats()
    env.rollout_device(KMAX, N.POLICY_ZERO, viol_count=vcnt, done_count=dcnt)
    counters, _ = env.read_stats()
    exact(counters, vcnt[:n].cpu().numpy(), dcnt[:n].cpu().numpy(), KMAX, "one launch of K_max")
    env.clear_stats()
    T = (1 << 22) + 3
    out = env.rollout_host(T, N.POLICY_ZERO, steps_per_launch=0)
    exact(out["counters"], out["violations"], out["episodes"], T, "host call of 2^22 + 3 steps")
    with pytest.raises(ValueError):
        env.rollout_device(KMAX + 1, N.POLICY_ZERO)
    with pytest.raises(ValueError):
        env.rollout_steps_device(KMAX + 1, KMAX + 1, N.POLICY_ZERO)
    env.close()
