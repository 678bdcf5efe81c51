"""NIG_POLICY_MLP: a learned MLP actor evaluated by tcgen05 MMAs inside the fused rollout (rollout_mlp_kernel).

Two separate checks:
1. the network: nig_selftest_mlp (the rollout's own device function and 128-row tiling) against an fp64 forward pass of the
   bf16-rounded network, to a tolerance derived from bf16 rounding (see fp64_forward); NaN / inf rows; row independence;
   determinism;
2. the rollout: the CPU oracle stepped one tick at a time with the actions nig_selftest_mlp returns for the oracle's current
   states, compared bit for bit after every launch (states, episode words, done latches, per-env sums and counts, the
   statistics window with extrema) -- the bit-exact contract downstream of the action.
"""
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

from util import KINDS, Track, adversarial, assert_bits_equal, compare_state, compare_stats

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def mods():
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    from oracle import oracle as O
    return ni, N, O, torch


def make_mlp(ni, rng, S, A, hidden, tanh=True, norm=None):
    """Random actor; the output bias is drawn from +-1 so that a dropped bias exceeds the tolerance."""
    dims = [S] + list(hidden) + [A]
    ws = [rng.uniform(-1, 1, (dims[k + 1], dims[k])).astype(np.float32) * np.float32(1.7 / np.sqrt(dims[k]))
          for k in range(len(dims) - 1)]
    bs = [rng.uniform(-0.2, 0.2, dims[k + 1]).astype(np.float32) for k in range(len(dims) - 2)]
    bs.append(rng.uniform(-1, 1, A).astype(np.float32))
    mean, std = (None, None) if norm is None else norm
    return ni.MLPPolicy(ws, bs, "tanh" if tanh else "identity", obs_mean=mean, obs_std=std)


def fp64_forward(pol, obs, weight_rounding=False):
    """Reference forward pass of the bf16-rounded network in fp64 and a bound on |device - reference| per output.

    The input x0 = bf16((s - mean) * inv_std) is computed identically on both sides (fp32, round to nearest). Per layer,
    with e the bound on the input error: |dz| <= |W| e + g_K |W| (|x| + e) (fp32 accumulation, g_K = (K + 2) 2^-24), plus
    2^-24 |z + b| for the fp32 bias add; ReLU and tanh are 1-Lipschitz. The next layer's input is rounded to bf16 on both
    sides: the two roundings of nearly equal values can land on neighbouring bf16 numbers, so the error grows by 2^-8 of
    each side's magnitude (2^-8 relative per element, then carried through sum |W| |x| of the following layers).
    weight_rounding=True also bounds a forward pass with unrounded fp32 weights and inputs (torch's own): 2^-8 |W| |x|."""
    from neorl_industrial.policies import bf16_round
    x = bf16_round(pol._input(obs)).astype(np.float64)
    e = np.zeros_like(x)
    n_layers = len(pol.weights)
    with np.errstate(invalid="ignore", over="ignore"):
        for k, (w, b) in enumerate(zip(pol.weights, pol.biases)):
            wb = bf16_round(w).astype(np.float64)
            aw = np.abs(wb)
            z = x @ wb.T
            ax = np.abs(x) + e
            g = (w.shape[1] + 2) * 2.0 ** -24
            dz = e @ aw.T + g * (ax @ aw.T)
            if weight_rounding:
                dz += 2.0 ** -8 * (ax @ aw.T) * 2 + (2.0 ** -8 * ax) @ aw.T
            y = z + b.astype(np.float64)
            dz += 2.0 ** -24 * np.abs(y)
            if k < n_layers - 1:
                y = np.where(y < 0, 0.0, y)
                x_next = bf16_round(y.astype(np.float32)).astype(np.float64)
                e = dz + 2.0 ** -8 * (np.abs(y) + dz) + 2.0 ** -8 * np.abs(y)
                x = x_next
            else:
                x, e = y, dz
    if pol.output_activation == "tanh":
        x = np.tanh(x)
    return x, e + 1e-6


def assert_within(dev, ref, bound, what):
    nan_ref, nan_dev = np.isnan(ref), np.isnan(dev)
    assert np.array_equal(nan_ref, nan_dev), f"{what}: NaN pattern differs ({np.count_nonzero(nan_ref != nan_dev)} elements)"
    ok = ~nan_ref
    inf = ok & np.isinf(ref)
    assert np.array_equal(dev[inf], ref[inf]), f"{what}: infinities differ"
    fin = ok & ~inf
    err = np.abs(dev[fin].astype(np.float64) - ref[fin])
    worst = np.argmax(err / bound[fin]) if err.size else 0
    assert (err <= bound[fin]).all(), (f"{what}: {np.count_nonzero(err > bound[fin])} of {err.size} outside the bound; worst "
                                       f"err {err[worst]:.3g} vs bound {bound[fin][worst]:.3g}")
    return float(err.max()) if err.size else 0.0, float(np.median(bound[fin])) if err.size else 0.0


NETS = [((64,), True, False), ((128, 128), False, True), ((256, 256), True, True), ((256, 64), False, False),
        ((64, 256), True, False), ((128,), False, True), ((256,), True, False), ((64, 64), False, True),
        ((64, 128), True, True), ((128, 64), True, False), ((128, 256), False, False), ((256, 128), False, True)]


# ---------------------------------------------------------------------------------------------------------------------
# 1. the network
@pytest.mark.parametrize("hidden,tanh,norm", NETS)
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_network_vs_fp64_forward(mods, name, hidden, tanh, norm):
    """nig_selftest_mlp == fp64 forward of the bf16-rounded network within the derived bound, for every env's S / A,
    widths 64 / 128 / 256, one and two hidden layers, both output activations, with and without normalisation. The
    observations are the env's own reset states moved by random steps (norm) or standard normals."""
    ni, N, O, torch = mods
    kind, n = KINDS[name], 4_099
    rng = np.random.default_rng(zlib.crc32(repr((name, hidden, tanh)).encode()))
    env = ni.NativeEnv(kind, n, device=0, seed=3)
    if norm:
        obs = env.reset_host()
        obs = obs + rng.normal(0, 1, obs.shape).astype(np.float32) * (np.abs(obs) * 0.05 + 0.1)
        mean, std = obs.mean(0).astype(np.float32), (obs.std(0) + 1e-3).astype(np.float32)
        pol = make_mlp(ni, rng, env.S, env.A, hidden, tanh, (mean, std))
    else:
        obs = rng.normal(0, 1, (n, env.S)).astype(np.float32)
        pol = make_mlp(ni, rng, env.S, env.A, hidden, tanh)
    obs = np.ascontiguousarray(obs, np.float32)
    env.set_mlp_policy(pol)
    dev = env.selftest_mlp(obs)
    ref, bound = fp64_forward(pol, obs)
    assert_within(dev, ref, bound, f"{name} {hidden}")
    assert_within(pol.predict(obs), ref, bound, f"{name} {hidden}: predict")    # predict is the same network
    env.close()


def test_from_torch_against_module(mods):
    """MLPPolicy.from_torch of a 256-256 tanh actor: the device equals the fp64 forward of the bf16 network within the bound,
    and the torch module's own fp32 forward within the bound widened by the rounding of weights and inputs."""
    ni, N, O, torch = mods
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(12, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(),
                              torch.nn.Linear(256, 3), torch.nn.Tanh())
    env = ni.NativeEnv(0, 1_000, device=0, seed=1)
    obs = env.reset_host()
    mean, std = obs.mean(0), obs.std(0) + 1.0
    pol = ni.MLPPolicy.from_torch(net, obs_mean=mean, obs_std=std)
    env.set_mlp_policy(pol)
    dev = env.selftest_mlp(obs)
    ref, bound = fp64_forward(pol, obs)
    assert_within(dev, ref, bound, "from_torch vs fp64")
    with torch.no_grad():
        t = net(torch.from_numpy(pol._input(obs))).numpy().astype(np.float64)
    _, wide = fp64_forward(pol, obs, weight_rounding=True)
    assert_within(dev, t, wide + bound, "from_torch vs the torch module")
    env.close()


def test_nan_inf_rows_rows_independent_and_deterministic(mods):
    """NaN / +-inf / huge observations give torch's NaN semantics in their own rows only; perturbing one row leaves every
    other row's actions bit-identical; two calls give identical bits."""
    ni, N, O, torch = mods
    rng = np.random.default_rng(5)
    n = 1_000
    env = ni.NativeEnv(2, n, device=0, seed=1)
    pol = make_mlp(ni, rng, env.S, env.A, (128, 128), False)
    env.set_mlp_policy(pol)
    obs = rng.normal(0, 1, (n, env.S)).astype(np.float32)
    clean = env.selftest_mlp(obs)
    assert_bits_equal(env.selftest_mlp(obs), clean, "second call")
    bad = obs.copy()
    rows = {3: np.nan, 130: np.inf, 131: -np.inf, 257: 1e30, 600: -1e30}
    for r, v in rows.items():
        bad[r, r % env.S] = v
    got = env.selftest_mlp(bad)
    other = np.setdiff1d(np.arange(n), list(rows))
    assert_bits_equal(got[other], clean[other], "rows next to NaN / inf / huge rows")
    ref, bound = fp64_forward(pol, bad)
    assert np.isnan(got[3]).all() and np.isnan(ref[3]).all()
    sel = np.array(sorted(rows))
    assert np.array_equal(np.isnan(got[sel]), np.isnan(ref[sel])), (got[sel], ref[sel])
    fin = np.isfinite(ref[sel]) & np.isfinite(got[sel])
    assert np.array_equal(np.sign(got[sel][fin]), np.sign(ref[sel][fin]))
    for r in range(0, n, 97):
        pert = obs.copy()
        pert[r] += 0.5
        out = env.selftest_mlp(pert)
        keep = np.arange(n) != r
        assert_bits_equal(out[keep], clean[keep], f"perturbing row {r}")
        assert not np.array_equal(out[r], clean[r])
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. the rollout against the oracle
def _start(ni, N, O, kind, n, *, seed, env_id_offset=0, max_episode_steps=None, auto_reset=True, constraints=None, threads=1):
    env = ni.NativeEnv(kind, n, device=0, seed=seed, env_id_offset=env_id_offset, max_episode_steps=max_episode_steps,
                       auto_reset=auto_reset, constraints=constraints)
    kw = {}
    if constraints is not None:
        kw = {"builtin": False, "extra_cons": [O.Con(c.kind, c.id, c.si, c.ai, c.coef, c.lo, c.hi, c.penalty, c.critical)
                                               for c in constraints]}
    orc = O.OracleEnv(kind, n, auto_reset=auto_reset, seed=seed, env_id0=env_id_offset, exp_mode=1,
                      max_episode_steps=max_episode_steps, threads=threads, **kw)
    assert_bits_equal(env.reset_host(), orc.reset(), "reset draw")
    return env, orc


def _adversarial_start(env, orc, O, kind, rng, auto_reset=True):
    n = orc.n
    st, ep_step = adversarial(O, kind, rng, orc.state.copy(), n, env.max_episode_steps) if n >= 400 else \
        (orc.state.copy(), np.zeros(n, np.int32))
    done = np.zeros(n, np.uint8) if auto_reset else (rng.random(n) < 0.05).astype(np.uint8)
    env.set_state_host(st, ep_step, np.zeros(n, np.int32), done)
    orc.state[:] = st
    orc.ep_step[:] = ep_step
    orc.ep_viol[:] = 0
    orc.done_latch[:] = done


def _run(env, orc, tr, N, torch, chunks, ncons, extrema, what):
    """One comparison per element of chunks: a launch of K steps, or a tuple of launches issued back to back (programmatic
    dependent launch lets the next one start while the previous one runs) and compared launch by launch."""
    n = orc.n
    for K in chunks:
        Ks = K if isinstance(K, tuple) else (K,)
        outs = [(env.empty(), env.empty(dtype=torch.int32), env.empty(dtype=torch.int32)) for _ in Ks]
        torch.cuda.synchronize()
        for k, (rsum, vcnt, dcnt) in zip(Ks, outs):
            env.rollout_device(k, N.POLICY_MLP, reward_sum=rsum, viol_count=vcnt, done_count=dcnt)
        torch.cuda.synchronize()
        for c, (k, (rsum, vcnt, dcnt)) in enumerate(zip(Ks, outs)):
            o_rs, o_v, o_d = tr.launch(k, lambda: env.selftest_mlp(orc.state))
            w = f"{what} after a {K}-step launch" if len(Ks) == 1 else f"{what}, launch {c} of {K} issued back to back"
            assert_bits_equal(rsum[:n].cpu().numpy(), o_rs, f"{w}: per-env reward sum")
            assert_bits_equal(vcnt[:n].cpu().numpy().astype(np.int64), o_v, f"{w}: per-env violation count")
            assert_bits_equal(dcnt[:n].cpu().numpy().astype(np.int64), o_d, f"{w}: per-env done count")
        compare_state(env, orc, w)
        counters, sums = env.read_stats()
        compare_stats(N, counters, sums, tr, ncons, extrema, w, env.read_extrema())
        env.clear_stats()
        tr.clear()


def _generic_cons(N, kind):
    """Re-ordered built-ins and an appended bound with an action term: CONS_GENERIC."""
    from neorl_industrial.vector import make_constraint
    spec = N.env_spec(kind)
    b = [make_constraint(N.CON_BUILTIN, cid=k, penalty=spec.constraints[k].penalty, critical=bool(spec.constraints[k].critical))
         for k in range(3)]
    lo, hi = (290.0, 330.0) if kind == 0 else (-0.3, 0.3)
    return [b[2], b[0], b[1], make_constraint(N.CON_BOUND, si=0, ai=0, coef=0.5, lo=lo, hi=hi, penalty=-7.0)]


CASES = [  # name, n, cons, auto_reset, episode cap, extrema, launches, (hidden, tanh) or None: 128-128 (grid 256-256) tanh
    ("reactor", 1_000, "default", True, None, True, (40, 7), None),
    ("reactor", 4_099, "generic", True, 30, False, (33, 1), None),
    ("reactor", 1, "default", True, 20, True, (45,), None),
    ("reactor", 1_000, "default", False, 25, True, (40,), None),
    ("grid", 1_000, "default", True, None, True, (20, 5), None),
    ("grid", 4_133, "generic", True, 15, True, (20,), None),
    ("grid", 1_000, "default", False, 15, False, (25,), None),
    ("robot", 1_000, "default", True, 30, True, (40, 3), None),
    ("robot", 1_000, "generic", False, 20, True, (30,), None),
    # one hidden layer, and identity outputs beyond +-1: the env's clip of the action
    ("reactor", 1_000, "default", True, None, True, (40,), ((64,), False)),
    ("grid", 1_000, "generic", True, 15, True, (20,), ((256,), False)),
    ("robot", 1_000, "default", True, 30, True, (30,), ((128,), True)),
    ("robot", 1_000, "generic", False, 20, False, (25,), ((64, 256), False)),
    # full tensor-memory occupancy on 148 SMs, two launches issued back to back: 2 CTAs per SM for two waves (256 columns),
    # and 1 CTA per SM holding all 512 columns, so that a CTA of the second launch waits in tcgen05.alloc behind the first
    ("reactor", 75_853, "default", True, 40, True, ((5, 3),), None),
    ("grid", 37_965, "default", True, 30, True, ((4, 3),), None),
]


def _case_id(i, case):
    """pytest's default id of the first seven fields, then the network where it is not the default one."""
    name, n, cons, auto_reset, cap, extrema, _, net = case
    cid = f"{name}-{n}-{cons}-{auto_reset}-{cap}-{extrema}-chunks{i}"
    return cid if net is None else f"{cid}-{'x'.join(map(str, net[0]))}-{'tanh' if net[1] else 'identity'}"


@pytest.mark.parametrize("name,n,cons,auto_reset,cap,extrema,chunks,net", CASES,
                         ids=[_case_id(i, c) for i, c in enumerate(CASES)])
def test_rollout_vs_oracle(mods, name, n, cons, auto_reset, cap, extrema, chunks, net):
    """The fused MLP rollout == the oracle driven by nig_selftest_mlp, bit for bit after every launch, from the adversarial
    start population, for CONS_DEFAULT and CONS_GENERIC, with and without auto-reset, with episode caps below K, one and two
    hidden layers, identity outputs clipped by the env, and populations that fill every SM's tensor memory."""
    ni, N, O, torch = mods
    kind = KINDS[name]
    cs = None if cons == "default" else _generic_cons(N, kind)
    env, orc = _start(ni, N, O, kind, n, seed=21, env_id_offset=5, max_episode_steps=cap, auto_reset=auto_reset, constraints=cs,
                      threads=O.max_threads() if n > 10_000 else 1)
    rng = np.random.default_rng(n)
    _adversarial_start(env, orc, O, kind, rng, auto_reset)
    hidden, tanh = net or ((128, 128) if name != "grid" else (256, 256), True)
    env.set_mlp_policy(make_mlp(ni, rng, env.S, env.A, hidden, tanh))
    if not tanh:
        a = env.selftest_mlp(orc.state)
        assert (np.abs(a) > 1).mean() > 0.05, "the identity network's actions should exercise the clip"
    env.track_extrema(extrema)
    tr = Track(orc, name)
    _run(env, orc, tr, N, torch, chunks, 3 if cs is None else 4, extrema, f"{name} n={n} {cons}")
    env.close()


def test_rollout_pair_size_vs_oracle(mods):
    """131,072 + 4,099 reactor envs (the size at which the uniform policy takes the pair kernel): one launch, bit for bit."""
    ni, N, O, torch = mods
    n = 131_072 + 4_099
    env, orc = _start(ni, N, O, 0, n, seed=8, max_episode_steps=40, threads=O.max_threads())
    rng = np.random.default_rng(0)
    _adversarial_start(env, orc, O, 0, rng)
    env.set_mlp_policy(make_mlp(ni, rng, env.S, env.A, (64, 64), True))
    env.track_extrema(True)
    _run(env, orc, Track(orc, "reactor"), N, torch, (12,), 3, True, "pair-size population")
    env.close()


def test_safety_wrapper_rollout(mods):
    """env.rollout(T, mlp) through SafetyWrapper (an appended bound with an action term) == the oracle with that set."""
    ni, N, O, torch = mods
    from neorl_industrial.safety import SafetyWrapper
    n, T, K = 500, 90, 32
    base = ni.ChemicalReactorEnv(num_envs=n, seed=4, env_id_offset=3, max_episode_steps=40)
    env = SafetyWrapper(base, [ni.BoundConstraint("t_band", 0, 300, 330, penalty=-30, action_index=0, action_coef=0.2)])
    cs = base._native_constraints()
    orc = O.OracleEnv(O.REACTOR, n, seed=4, env_id0=3, exp_mode=1, max_episode_steps=40, builtin=False,
                      extra_cons=[O.Con(c.kind, c.id, c.si, c.ai, c.coef, c.lo, c.hi, c.penalty, c.critical) for c in cs])
    orc.reset()
    pol = make_mlp(ni, np.random.default_rng(2), 12, 3, (64, 128), True)
    res = env.rollout(T, pol, steps_per_launch=K, reset=True)
    ev = ni.NativeEnv(0, n, device=0, seed=0)
    ev.set_mlp_policy(pol)
    tr = Track(orc, "reactor")
    total = None
    for c0 in range(0, T, K):
        part, _, _ = tr.launch(min(K, T - c0), lambda: ev.selftest_mlp(orc.state))
        total = part if total is None else (total + part).astype(np.float32)
    assert_bits_equal(res["obs"], orc.state, "final state")
    assert_bits_equal(res["reward_sum"], total, "reward_sum")
    assert res["stats"]["violations"] == orc.stats[5] and res["stats"]["episodes"] == orc.stats[1] > 0
    ev.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. the host-side paths: slicing, graphs, host buffers, re-setting the network
def _steps_run(ni, N, torch, monkeypatch, slices, graph, nets, n=65_536 + 4_099):
    monkeypatch.setenv("NIG_HOST_SLICES", str(slices))
    monkeypatch.setenv("NIG_STEPS_GRAPH", "1" if graph else "0")
    env = ni.NativeEnv(0, n, device=0, seed=77, max_episode_steps=50)
    env.reset_host()
    env.track_extrema(True)
    rs = env.empty()
    out = []
    for pol in nets:
        env.set_mlp_policy(pol)
        for _ in range(2):                                 # the second identical call captures (or replays) the graph
            env.rollout_steps_device(70, 32, N.POLICY_MLP, reward_sum=rs)
        torch.cuda.synchronize()
        out.append((env.get_state_host(), rs[:n].cpu().numpy().copy(), env.read_stats(), env.read_extrema()))
    env.close()
    return out


def test_rollout_steps_slices_graphs_and_network_changes(mods, monkeypatch):
    """nig_rollout_steps with 1 vs 8 env slices and graph replay vs NIG_STEPS_GRAPH=0 give identical bits, also after the
    network is re-set with the same shape and then with a different shape between calls (a replay must not run the old
    network)."""
    ni, N, O, torch = mods
    rng = np.random.default_rng(9)
    a = make_mlp(ni, rng, 12, 3, (128, 128), True)
    b = make_mlp(ni, rng, 12, 3, (128, 128), True)
    c = make_mlp(ni, rng, 12, 3, (256,), False)
    runs = {(s, g): _steps_run(ni, N, torch, monkeypatch, s, g, [a, b, c]) for s, g in [(8, True), (8, False), (1, False)]}
    ref = runs[(1, False)]
    for key, got in runs.items():
        for phase, (x, y) in enumerate(zip(got, ref)):
            w = f"slices/graph {key}, network {phase}"
            for k in range(4):
                assert_bits_equal(x[0][k], y[0][k], f"{w}: state part {k}")
            assert_bits_equal(x[1], y[1], f"{w}: reward sum")
            assert np.array_equal(x[2][0], y[2][0]) and np.allclose(x[2][1], y[2][1], rtol=1e-12), w
            assert x[3] == y[3], w
    assert not np.array_equal(ref[0][1], ref[1][1]) and not np.array_equal(ref[1][1], ref[2][1])
    # re-setting the network on a handle whose graph was captured == a fresh handle that only ever had the last network,
    # from the same state and tick: states, per-env rewards, statistics and extrema (8 slices, graph replay)
    monkeypatch.setenv("NIG_HOST_SLICES", "8")
    monkeypatch.setenv("NIG_STEPS_GRAPH", "1")
    n = 65_536 + 4_099
    env = ni.NativeEnv(0, n, device=0, seed=77, max_episode_steps=50)
    env.reset_host()
    env.track_extrema(True)
    rs = env.empty()
    for pol in (a, b):
        env.set_mlp_policy(pol)
        for _ in range(2):
            env.rollout_steps_device(70, 32, N.POLICY_MLP, reward_sum=rs)
    torch.cuda.synchronize()
    fresh = ni.NativeEnv(0, n, device=0, seed=77, max_episode_steps=50)
    st = env.get_state_host()
    fresh.set_state_host(*st)
    env.set_state_host(*st)        # importing an episode step restarts the return accumulator: the same on both handles
    fresh.set_tick(env.tick, env.epoch)
    fresh.track_extrema(True)
    fresh.set_mlp_policy(c)
    env.set_mlp_policy(c)
    env.clear_stats()
    rs_f = fresh.empty()
    for _ in range(2):
        env.rollout_steps_device(70, 32, N.POLICY_MLP, reward_sum=rs)
        fresh.rollout_steps_device(70, 32, N.POLICY_MLP, reward_sum=rs_f)
    torch.cuda.synchronize()
    for k, (x, y) in enumerate(zip(env.get_state_host(), fresh.get_state_host())):
        assert_bits_equal(x, y, f"re-set network vs fresh handle: state part {k}")
    assert_bits_equal(rs[:n].cpu().numpy(), rs_f[:n].cpu().numpy(), "re-set network vs fresh handle: reward sum")
    (c1, s1), (c2, s2) = env.read_stats(), fresh.read_stats()
    assert np.array_equal(c1, c2) and np.allclose(s1, s2, rtol=1e-12, atol=0), (c1, c2, s1, s2)
    assert env.read_extrema() == fresh.read_extrema() and env.read_extrema()[0] is not None
    env.close(); fresh.close()


def test_single_env_make_rollout(mods):
    """Population 1 through the single-env API: ni.make(...).rollout(T, mlp) == the oracle driven by nig_selftest_mlp."""
    ni, N, O, torch = mods
    T, K = 130, 64
    env = ni.make("RobotAssembly-v0", seed=12)
    assert not env.batched and env.num_envs == 1 and not env.auto_reset
    orc = O.OracleEnv(O.ROBOT, 1, seed=12, exp_mode=1, auto_reset=False)
    orc.reset()
    pol = make_mlp(ni, np.random.default_rng(12), 24, 7, (128, 64), True)
    res = env.rollout(T, pol, steps_per_launch=K, reset=True)
    ev = ni.NativeEnv(2, 1, device=0, seed=0)
    ev.set_mlp_policy(pol)
    tr = Track(orc, "robot")
    total = None
    for c0 in range(0, T, K):
        part, _, _ = tr.launch(min(K, T - c0), lambda: ev.selftest_mlp(orc.state))
        total = part if total is None else (total + part).astype(np.float32)
    assert_bits_equal(np.asarray(res["obs"]).reshape(1, -1), orc.state, "final state")
    assert_bits_equal(np.asarray(res["reward_sum"]).reshape(1), total, "reward_sum")
    assert res["stats"]["steps"] == orc.stats[0] > 0 and res["stats"]["episodes"] == orc.stats[1]
    ev.close(); env.close()


def test_rollout_host_direct_vs_staged(mods, monkeypatch):
    """nig_rollout_host with NIG_POLICY_MLP: the direct (page-locked) and staged paths, sliced, give identical bits."""
    ni, N, O, torch = mods
    n, rng = 40_000, np.random.default_rng(4)
    pol = make_mlp(ni, rng, 24, 7, (64, 64), True)
    outs = []
    for direct in ("3", "0"):
        monkeypatch.setenv("NIG_HOST_DIRECT", direct)
        env = ni.NativeEnv(2, n, device=0, seed=31, max_episode_steps=40)
        env.set_mlp_policy(pol)
        out = env.rollout_host(150, N.POLICY_MLP, steps_per_launch=64, reset_first=True)
        outs.append({k: np.array(v, copy=True) for k, v in out.items() if isinstance(v, np.ndarray)})
        env.close()
    for k in outs[0]:
        if k == "sums":          # fp64 sums are accumulated with atomics in no fixed order
            np.testing.assert_allclose(outs[0][k], outs[1][k], rtol=1e-12, atol=0)
        else:
            assert_bits_equal(outs[0][k], outs[1][k], f"rollout_host direct vs staged: {k}")
    assert outs[0]["episodes"].sum() > 0


# ---------------------------------------------------------------------------------------------------------------------
# 4. public entry points, dispatch witness, errors
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_public_entry_points(mods, name):
    """env.rollout(1000, MLPPolicy.from_torch(actor)) and evaluate_policy_device(env, 1000, policy=mlp) for every env; the
    network is uploaded once per network object."""
    ni, N, O, torch = mods
    from neorl_industrial.rollouts import evaluate_policy_device
    env = ni.make({"reactor": "ChemicalReactor-v0", "grid": "PowerGrid-v0", "robot": "RobotAssembly-v0"}[name], num_envs=2_048)
    torch.manual_seed(1)
    S, A = env.native.S, env.native.A
    actor = torch.nn.Sequential(torch.nn.Linear(S, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(),
                                torch.nn.Linear(256, A), torch.nn.Tanh())
    mlp = ni.MLPPolicy.from_torch(actor)
    res = env.rollout(1000, mlp, reset=True)
    assert res["stats"]["steps"] == 2_048 * 1000 and np.isfinite(res["reward_sum"]).all()
    out = evaluate_policy_device(env, 1000, policy=mlp)
    for k in ("return_mean", "return_std", "return_min", "return_max", "length_mean", "safety_violations",
              "constraint_satisfaction_rate", "success_rate", "episodes", "steps"):
        assert k in out, k
    assert out["steps"] == 2_048 * 1000 and out["episodes"] > 0 and out["return_min"] <= out["return_max"]
    assert env.native._mlp is mlp
    env.close()


WITNESS = r"""
import sys, numpy as np
sys.path[:0] = [{root!r}, {root!r} + "/tests", {root!r} + "/neorl-industrial-gym_b200"]
import torch
import neorl_industrial as ni
from neorl_industrial import _native as N
from util import kernel_names, template_args
rng = np.random.default_rng(0)
for kind, n in ((0, 131_072 + 4_099), (0, 1_000), (1, 4_133), (2, 1_000)):
    env = ni.NativeEnv(kind, n, device=0, seed=1)
    env.reset_host()
    ws = [rng.normal(0, .1, (64, env.S)).astype(np.float32), rng.normal(0, .1, (env.A, 64)).astype(np.float32)]
    env.set_mlp_policy(ni.MLPPolicy(ws))
    names = kernel_names(torch, lambda: env.rollout_device(8, N.POLICY_MLP))
    print(kind, n, sorted(x for x in names if "rollout" in x))
    assert template_args(names, "rollout_mlp_kernel"), names
    assert not [x for x in names if "rollout_kernel" in x or "pair_kernel" in x or "grid_kernel" in x], names
    env.close()
print("witness ok")
"""


def test_dispatch_witness(mods):
    """rollout_mlp_kernel runs for every env, also at sizes and switch values that select the pair kernel (reactor 135,171
    envs, NIG_ROLLOUT_PAIR=1, NIG_ROLLOUT_BLOCK=32) or the grid-fast kernel (PowerGrid 4,133) for other policies. Recorded in
    a child process (profiler sessions early in a suite can leave later ones empty)."""
    envs = dict(os.environ, NIG_ROLLOUT_PAIR="1", NIG_ROLLOUT_BLOCK="32", NIG_GRID_FAST="1")
    out = subprocess.run([sys.executable, "-c", WITNESS.format(root=ROOT)], capture_output=True, text=True, env=envs,
                         timeout=600)
    assert out.returncode == 0 and "witness ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


def test_error_paths(mods):
    ni, N, O, torch = mods
    import ctypes as C
    env = ni.NativeEnv(0, 256, device=0, seed=1)
    env.reset_host()
    with pytest.raises(ValueError, match="needs a network"):
        env.rollout_device(4, N.POLICY_MLP)
    with pytest.raises(ValueError, match="needs a network"):
        env.rollout_steps_device(8, 4, N.POLICY_MLP)
    with pytest.raises(ValueError, match="no network"):
        env.selftest_mlp(np.zeros((4, 12), np.float32))
    rng = np.random.default_rng(0)
    pol = make_mlp(ni, rng, 12, 3, (64,), True)
    env.set_mlp_policy(pol)
    env.rollout_device(4, N.POLICY_MLP)
    with pytest.raises(NotImplementedError):                       # teacher-forced noise with an in-kernel policy
        env.rollout_device(4, N.POLICY_MLP, noise=env.empty(rows=4 * 2))
    with pytest.raises(NotImplementedError):
        env.rollout_host(8, N.POLICY_MLP, noise=np.zeros((8, 2, 256), np.float32))
    with pytest.raises(NotImplementedError):
        env.dataset_size(10, 10, N.POLICY_MLP, N.PolicyParams())
    with pytest.raises(NotImplementedError):
        out = {"observations": env.empty(rows=12), "actions": env.empty(rows=3), "rewards": env.empty(rows=1),
               "terminals": env.empty(rows=1, dtype=torch.uint8)}
        env.dataset_device(10, 10, N.POLICY_MLP, N.PolicyParams(), out, 100)
    with pytest.raises(ValueError, match="env needs"):             # robot network on a reactor handle
        env.set_mlp_policy(make_mlp(ni, rng, 24, 7, (64,), True))
    m = pol.native_struct()
    for field, value in (("n_hidden", 3), ("n_hidden", 0), ("output_activation", 2)):
        bad = pol.native_struct()
        setattr(bad, field, value)
        with pytest.raises(ValueError):
            N.check(N.lib().nig_set_mlp_policy(env._h, C.byref(bad)))
    bad = pol.native_struct()
    bad.hidden[0] = 96
    with pytest.raises(ValueError, match="hidden width"):
        N.check(N.lib().nig_set_mlp_policy(env._h, C.byref(bad)))
    del m
    env.rollout_device(4, N.POLICY_MLP)                            # the rejected calls left the network in place
    torch.cuda.synchronize()
    env.close()
