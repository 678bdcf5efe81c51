"""GPU tests added in round 2: the invariant-specialised reactor rollout loop against the oracle from adversarial entry
states, the episode-return bookkeeping across mixed nig_step / nig_rollout use, the exact-size host outputs of the
zero-copy step path, seeded resets."""
import ctypes as C

import numpy as np
import pytest

from util import KINDS, Track, assert_bits_equal, compare_stats

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    from oracle import oracle as O
    return ni, N, O, torch


def _compare(env, orc, N, what):
    st, ep_step, ep_viol, done = env.get_state_host()
    assert_bits_equal(st, orc.state, f"{what}: state")
    assert_bits_equal(ep_step, orc.ep_step, f"{what}: episode step")
    assert_bits_equal(ep_viol, orc.ep_viol, f"{what}: episode violations")
    assert_bits_equal(done, orc.done_latch, f"{what}: done latch")
    counters, _ = env.read_stats()
    assert counters[:6].tolist() == orc.stats[:6].tolist(), (what, counters[:8], orc.stats[:8])
    assert counters[N.ST_CON0:N.ST_CON0 + 3].tolist() == orc.stats[8:11].tolist(), what


def test_reactor_fast_loop_from_adversarial_entry_states(mods):
    """The specialised loop is entered per warp only when every env of the warp satisfies its invariants; these populations
    mix warps that do with warps that do not (tripped e-stop, alarm set, fractional latch values, -0.0 flags, over-limit
    temperature / pressure, odd catalyst values, episodes about to be truncated, a NaN) -- every result must still be the
    oracle's, bit for bit, including the states the loop never saw."""
    ni, N, O, torch = mods
    rng = np.random.default_rng(5)
    n, K = 4096 + 37, 48
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=21)
    orc = O.OracleEnv(O.REACTOR, n, seed=21, exp_mode=1)
    s0 = env.reset_host()
    assert_bits_equal(s0, orc.reset(), "reset")
    st = s0.copy()
    ep_step = np.zeros(n, np.int32)
    # warp-sized groups of special cases (one odd env spoils its whole warp; whole warps of them too)
    def some(k):
        return rng.choice(n, k, replace=False)
    st[some(40), 8] = 1.0                      # e-stop already tripped
    st[some(40), 9] = 1.0                      # alarm latched (still inside the invariant)
    st[some(10), 8] = 0.3                      # fractional latch values the reference would carry along unchanged
    st[some(10), 9] = 0.7
    st[some(10), 8] = -0.0
    st[some(10), 9] = -0.0
    st[some(30), 0] = rng.uniform(350.0, 356.0, 30).astype(np.float32)     # over the temperature limit: critical shutdown
    st[some(30), 1] = rng.uniform(5.0e5, 5.2e5, 30).astype(np.float32)     # around the pressure limit
    st[some(10), 0] = 150.0                    # outside the loop's 200 .. 350 K entry range
    st[some(10), 5] = rng.choice([0.0, 1e-35, 49.0, 50.0, 3e30], 10).astype(np.float32)
    st[some(5), 4] = 0.0
    st[some(3), 0] = np.nan
    ep_step[some(200)] = rng.integers(440, 500, 200)                         # truncation inside the launch
    st[32 * 5:32 * 6, 8] = 1.0                 # one whole warp outside the invariant
    env.set_state_host(st, ep_step, np.zeros(n, np.int32), np.zeros(n, np.uint8))
    orc.state[:] = st
    orc.ep_step[:] = ep_step
    for chunk in (K, 17, 1, 64):
        env.rollout_device(chunk, N.POLICY_UNIFORM)
        O.rollout(orc, chunk, O.POLICY_UNIFORM)
        torch.cuda.synchronize()
        _compare(env, orc, N, f"after a {chunk}-step launch")
    env.close()


@pytest.mark.parametrize("shape", ["1", "2", "3", "4", "0"])
def test_grid_fast_loop_from_adversarial_entry_states(mods, monkeypatch, shape):
    """PowerGrid-v0: the dedicated lean rollout kernel (in-place step, min / max trees for the voltage ranges, max / min
    clamps, 8 x replicated normal table, rank-dealt cooperative reset) enters its loop per warp only when every env of the
    warp satisfies the invariants; these populations mix such warps with warps holding out-of-range / non-finite / signed-zero
    states and episodes about to be truncated. Everything must be the oracle's, bit for bit, for every CTA shape and for the
    generic kernel (NIG_GRID_FAST=0) alike; per-env sums, counters and episode statistics included."""
    ni, N, O, torch = mods
    monkeypatch.setenv("NIG_GRID_FAST", shape)
    rng = np.random.default_rng(11)
    n, K = 4096 + 37, 40
    env = ni.NativeEnv(N.ENV_POWER_GRID, n, device=0, seed=33, env_id_offset=96)
    orc = O.OracleEnv(O.GRID, n, seed=33, env_id0=96, exp_mode=1)
    s0 = env.reset_host()
    assert_bits_equal(s0, orc.reset(), "reset")
    st = s0.copy()
    ep_step = np.zeros(n, np.int32)
    def some(k):
        return rng.choice(n, k, replace=False)
    st[some(40), 0] = rng.uniform(-1.2, 1.2, 40).astype(np.float32)       # frequency: inside, at and beyond both limits
    st[some(6), 0] = np.array([0.5, -0.5, 1.0, -1.0, -0.0, 0.49999997], np.float32)
    i = some(40); st[i, 1 + rng.integers(0, 8, 40)] = rng.uniform(0.88, 1.12, 40).astype(np.float32)   # voltages around every threshold
    i = some(8); st[i, 1 + rng.integers(0, 8, 8)] = np.array([0.9, 0.95, 1.05, 1.1, 0.94999999, 1.0500001, 0.3, 2.5], np.float32)
    i = some(30); st[i, 9 + rng.integers(0, 8, 30)] = rng.choice([0.0, -0.0, 100.0, 99.5, 0.4, 100.5, -3.0, 1e-30], 30).astype(np.float32)
    i = some(20); st[i, 17 + rng.integers(0, 8, 20)] = rng.choice([0.0, -0.0, 1e-20, 0.3, 1e30, 3e38, -2.0], 20).astype(np.float32)
    i = some(10); st[i, 25 + rng.integers(0, 7, 10)] = rng.choice([0.0, -0.0, 3e38, -3e38, np.inf], 10).astype(np.float32)
    i = some(6); st[i, rng.integers(0, 32, 6)] = np.nan
    i = some(4); st[i, 17 + rng.integers(0, 8, 4)] = np.inf
    w = 32 * 7                                    # one warp with zero imbalance and zero frequency: the division guard fails
    st[w:w + 32, 0] = 0.0; st[w:w + 32, 9:17] = 50.0; st[w:w + 32, 17:25] = 50.0
    ep_step[some(300)] = rng.integers(950, 1000, 300)                      # truncation inside the launch
    env.set_state_host(st, ep_step, np.zeros(n, np.int32), np.zeros(n, np.uint8))
    orc.state[:] = st
    orc.ep_step[:] = ep_step
    rsum, vcnt, dcnt = env.empty(), env.empty(dtype=torch.int32), env.empty(dtype=torch.int32)
    for chunk in (K, 17, 1, 64):
        env.rollout_device(chunk, N.POLICY_UNIFORM, reward_sum=rsum, viol_count=vcnt, done_count=dcnt)
        o_rs = O.rollout(orc, chunk, O.POLICY_UNIFORM, want_reward_sum=True)
        torch.cuda.synchronize()
        _compare(env, orc, N, f"after a {chunk}-step launch")
        g_rs = rsum[:n].cpu().numpy()
        both_nan = np.isnan(g_rs) & np.isnan(o_rs)       # (NaN states injected above: the payload / sign of a NaN sum is not specified)
        assert_bits_equal(np.where(both_nan, 0, g_rs), np.where(both_nan, 0, o_rs), f"per-env reward sum of a {chunk}-step launch")
    env.close()


@pytest.mark.parametrize("auto_reset,mode", [(True, "1"), (False, "1"), (True, "2"), (True, "3"), (False, "6"), (True, "6"),
                                             (True, None), (False, None), (True, "4"), (False, "4"), (True, "0"), (False, "0")])
def test_grid_persistent_step_kernel_from_adversarial_states_and_actions(mods, monkeypatch, auto_reset, mode):
    """PowerGrid-v0 single step at a population large enough for the dedicated persistent kernel (lean in-place step with
    per-step guards, generic step_core as the per-warp fallback): out-of-range / non-finite / signed-zero states, NaN /
    infinite / over-range actions, generation-limit violations, envs on the brink of truncation, done latches (auto_reset
    off): rewards, flags, violation masks, states, episode words and counters equal to the oracle's, bit for bit, step after
    step, with the statistics window (episode statistics and fp64 return sums too) after every step; and to the one-tile
    kernel (NIG_GRID_STEP=0) through the same oracle. The dedicated kernel runs from three tiles per resident CTA: with the
    default shape (256 threads, two CTAs per SM) from 888 tiles = 227,073 envs on 148 SMs (test_gpu_step_flavours.py's
    dispatch witness checks that these n reach it)."""
    ni, N, O, torch = mods
    if mode is None:                                   # unset: the default shape, as "1"
        monkeypatch.delenv("NIG_GRID_STEP", raising=False)
    else:
        monkeypatch.setenv("NIG_GRID_STEP", mode)      # CTA shape / table replication of the dedicated kernel, "0": off
    rng = np.random.default_rng(17)
    n, T = 262_147, 7      # 1,025 tiles of 256 envs (1,366 of 192, 683 of 384, 2,049 of 128): every shape's dedicated kernel
    env = ni.NativeEnv(N.ENV_POWER_GRID, n, device=0, seed=5, env_id_offset=3, auto_reset=auto_reset)
    orc = O.OracleEnv(O.GRID, n, seed=5, env_id0=3, exp_mode=1, auto_reset=auto_reset, threads=O.max_threads())
    s0 = env.reset_host()
    assert_bits_equal(s0, orc.reset(), "reset")
    st = s0.copy()
    ep_step = np.zeros(n, np.int32)
    def some(k):
        return rng.choice(n, k, replace=False)
    st[some(400), 0] = rng.uniform(-1.2, 1.2, 400).astype(np.float32)
    st[some(6), 0] = np.array([0.5, -0.5, 1.0, -1.0, -0.0, np.inf], np.float32)
    i = some(400); st[i, 1 + rng.integers(0, 8, 400)] = rng.uniform(0.88, 1.12, 400).astype(np.float32)
    i = some(8); st[i, 1 + rng.integers(0, 8, 8)] = np.array([0.9, 0.95, 1.05, 1.1, 0.3, 2.5, np.inf, -1.0], np.float32)
    i = some(300); st[i, 9 + rng.integers(0, 8, 300)] = rng.choice([0.0, -0.0, 100.0, 99.5, 0.4, 100.5, -3.0, 1e-30], 300).astype(np.float32)
    i = some(200); st[i, 17 + rng.integers(0, 8, 200)] = rng.choice([0.0, -0.0, 1e-20, 0.3, 1e30, 3e38, -2.0, np.inf], 200).astype(np.float32)
    i = some(100); st[i, 25 + rng.integers(0, 7, 100)] = rng.choice([0.0, -0.0, 3e38, -3e38, np.inf], 100).astype(np.float32)
    i = some(60); st[i, rng.integers(0, 32, 60)] = np.nan
    w = 32 * 77
    st[w:w + 32, 0] = 0.0; st[w:w + 32, 9:17] = 50.0; st[w:w + 32, 17:25] = 50.0
    ep_step[some(3000)] = rng.integers(996, 1000, 3000)
    env.set_state_host(st, ep_step, np.zeros(n, np.int32), np.zeros(n, np.uint8))
    orc.state[:] = st
    orc.ep_step[:] = ep_step
    tr = Track(orc, "grid")
    dev = env.torch_device()
    rew, fl, vm = env.empty(), env.empty(dtype=torch.uint8), env.empty(dtype=torch.uint8)
    episodes = 0
    for t in range(T):
        a = rng.uniform(-1.3, 1.3, (n, env.A)).astype(np.float32)
        i = some(50); a[i, rng.integers(0, 8, 50)] = rng.choice([np.nan, np.inf, -np.inf, -0.0, 5.0], 50).astype(np.float32)
        if t == 0:
            a[w:w + 32] = 0.0
        d_a = torch.zeros((env.A, env.pitch), dtype=torch.float32, device=dev)
        d_a[:, :n] = torch.from_numpy(np.ascontiguousarray(a.T)).to(dev)
        env.step_device(d_a, reward=rew, flags=fl, viol_mask=vm)
        torch.cuda.synchronize()
        _, o_r, o_fl, o_vm = tr.step(a, want_next_obs=False)
        assert_bits_equal(fl[:n].cpu().numpy(), o_fl, f"flags t={t}")
        assert_bits_equal(vm[:n].cpu().numpy(), o_vm, f"viol t={t}")
        g_r = rew[:n].cpu().numpy()
        both_nan = np.isnan(g_r) & np.isnan(o_r)
        assert_bits_equal(np.where(both_nan, 0, g_r), np.where(both_nan, 0, o_r), f"reward t={t}")
        # (a NaN that flows through an addition keeps its payload on x86 and becomes the canonical NaN on the GPU: compare
        #  NaN-ness there, bits everywhere else)
        g_st = env.get_state_host()[0]
        nan_both = np.isnan(g_st) & np.isnan(orc.state)
        keep = orc.state.copy()
        orc.state[nan_both] = g_st[nan_both]
        _compare(env, orc, N, f"t={t}")
        orc.state[:] = keep
        counters, sums = env.read_stats()
        compare_stats(N, counters, sums, tr, 3, False, f"statistics t={t}", reward_sum=False)
        episodes += int(counters[N.ST_EPISODES])
        env.clear_stats()
        tr.clear()
    assert episodes > 0
    env.close()


def test_reactor_fast_loop_without_auto_reset_and_sharded(mods):
    """auto_reset off never enters the specialised loop (latches instead); shards keyed by global env id agree with the
    unsharded run whichever loop they took."""
    ni, N, O, torch = mods
    n, K = 2048, 96
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=4, auto_reset=False)
    orc = O.OracleEnv(O.REACTOR, n, seed=4, exp_mode=1, auto_reset=False)
    assert_bits_equal(env.reset_host(), orc.reset(), "reset")
    env.rollout_device(K, N.POLICY_UNIFORM)
    O.rollout(orc, K, O.POLICY_UNIFORM)
    torch.cuda.synchronize()
    _compare(env, orc, N, "no auto-reset")
    env.close()
    whole = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=9)
    whole.reset_host()
    whole.rollout_device(K, N.POLICY_UNIFORM)
    ref = whole.get_state_host()[0]
    for off, cnt in ((0, 700), (700, 1348)):
        e = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, cnt, device=0, seed=9, env_id_offset=off)
        e.reset_host()
        e.rollout_device(K, N.POLICY_UNIFORM)
        assert_bits_equal(e.get_state_host()[0], ref[off:off + cnt], f"shard at {off}")
        e.close()
    whole.close()


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_episode_returns_across_mixed_step_and_rollout_calls(mods, name):
    """One handle driven by alternating nig_step (host actions) and nig_rollout (the same actions drawn in-kernel) reports
    the finished-episode statistics of the all-rollout run: the running return of every episode lives in one per-env
    accumulator both kernels keep (ADVICE r01). Counters exact; fp64 sums to 1e-12 (atomics commute up to rounding)."""
    ni, N, O, torch = mods
    kind = KINDS[name]
    n = 3000
    # a 40-step episode cap so that every env finishes episodes inside the 106-step plan (reactor episodes run ~370 steps)
    a_env = ni.NativeEnv(kind, n, device=0, seed=33, max_episode_steps=40)
    b_env = ni.NativeEnv(kind, n, device=0, seed=33, max_episode_steps=40)
    orc = O.OracleEnv(kind, n, seed=33, exp_mode=1, max_episode_steps=40)
    a_env.reset_host(); b_env.reset_host(); orc.reset()
    plan = [("rollout", 9), ("step", 7), ("rollout", 30), ("step", 12), ("rollout", 5), ("step", 3), ("rollout", 40)]
    total = sum(k for _, k in plan)
    a_env.rollout_device(total, N.POLICY_UNIFORM)
    # ground truth from the oracle, one step at a time: per-env running return in the env's reward type (fp32 reactor,
    # fp64 grid / robot -- the accumulator type of the kernels), summed over finished episodes in fp64
    acc_t = np.float32 if name == "reactor" else np.float64
    run = np.zeros(n, acc_t)
    ret_sum = ret_sq = 0.0
    n_succ = len_sum = 0
    ep_len = np.zeros(n, np.int64)

    def oracle_step(act):
        nonlocal run, ret_sum, ret_sq, n_succ, len_sum, ep_len
        _, r, fl, _ = orc.step(act, want_next_obs=False)
        run = (run + r.astype(acc_t)).astype(acc_t)
        ep_len = ep_len + 1
        done = (fl & 3) > 0
        ret_sum += float(run[done].astype(np.float64).sum()); ret_sq += float((run[done].astype(np.float64) ** 2).sum())
        n_succ += int((run[done] > 0).sum()); len_sum += int(ep_len[done].sum())
        run[done] = 0; ep_len[done] = 0

    for how, k in plan:
        for _ in range(k):
            act = O.policy_actions(orc, O.POLICY_UNIFORM)
            if how == "step":
                b_env.step_host(act, want_obs=False)
            oracle_step(act)
        if how == "rollout":
            b_env.rollout_device(k, N.POLICY_UNIFORM)
    torch.cuda.synchronize()
    assert_bits_equal(a_env.get_state_host()[0], b_env.get_state_host()[0], "final states")
    assert_bits_equal(a_env.get_state_host()[0], orc.state, "final states vs oracle")
    ca, fa = a_env.read_stats()
    cb, fb = b_env.read_stats()
    assert ca[N.ST_EPISODES] >= 2 * n, "the plan must finish episodes"
    assert ca[:6].tolist() == orc.stats[:6].tolist()
    for what, (c, f) in {"all-rollout": (ca, fa), "mixed step / rollout": (cb, fb)}.items():
        assert c[:6].tolist() == orc.stats[:6].tolist(), what
        assert (c[N.ST_SUCCESSES], c[N.ST_EP_LEN_SUM]) == (n_succ, len_sum), (what, c[N.ST_SUCCESSES], n_succ, c[N.ST_EP_LEN_SUM], len_sum)
        # fp64 atomics commute up to rounding; the oracle hands its fp64 rewards (grid, robot) back rounded to fp32
        np.testing.assert_allclose(f[:2], [ret_sum, ret_sq], rtol=1e-11 if name == "reactor" else 1e-6, err_msg=what)
    np.testing.assert_allclose(fb[:2], fa[:2], rtol=1e-12)
    assert ca[N.ST_EP_LEN_SQ] == cb[N.ST_EP_LEN_SQ]
    # and with tracking switched off the step kernels leave the accumulator alone (documented behaviour)
    b_env.track_returns(False)
    b_env.clear_stats()
    act = O.policy_actions(orc, O.POLICY_UNIFORM)
    b_env.step_host(act, want_obs=False)
    cb2, fb2 = b_env.read_stats()
    assert cb2[N.ST_STEPS] == n and cb2[N.ST_EP_LEN_SUM] == 0 and fb2[0] == 0.0
    a_env.close(); b_env.close()


def test_set_state_restarts_the_episode_return(mods):
    ni, N, O, torch = mods
    n = 512
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=1)
    s0 = env.reset_host()
    env.rollout_device(20, N.POLICY_UNIFORM)                 # leaves partial returns in the accumulators
    env.set_state_host(s0, np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint8))
    env.clear_stats()
    env.set_tick(0)
    fresh = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=1)
    fresh.reset_host()
    fresh.set_state_host(s0, np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint8))
    fresh.set_tick(0, env.epoch)
    env.rollout_device(500, N.POLICY_UNIFORM)
    fresh.rollout_device(500, N.POLICY_UNIFORM)
    ca, fa = env.read_stats()
    cb, fb = fresh.read_stats()
    assert ca[N.ST_EPISODES] == cb[N.ST_EPISODES] > 0
    np.testing.assert_allclose(fa[:2], fb[:2], rtol=1e-12)
    env.close(); fresh.close()


@pytest.mark.parametrize("n", [1, 130])
def test_zero_copy_step_writes_nothing_past_n(mods, monkeypatch, n):
    """nig_step_host with page-locked buffers runs the kernel directly on them: a C caller may pack reward[n], flags[n],
    viol_mask[n], terminated[n], truncated[n], next_obs[n][S] back to back in ONE nig_host_alloc block -- nothing may be
    written past element n - 1 of any of them (ADVICE r01: the padding lanes up to pitch used to store 0.0 rewards / INACTIVE
    flags over the neighbours), whatever NIG_STEP_VEC says (the vector flavours store up to the pitch: AoS calls must not
    take them)."""
    ni, N, O, torch = mods
    S, A = 12, 3
    lib = N.lib()
    for vec in (None, "2", "4"):
        if vec is None:
            monkeypatch.delenv("NIG_STEP_VEC", raising=False)
        else:
            monkeypatch.setenv("NIG_STEP_VEC", vec)         # (read by nig_create)
        env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=2)
        env.reset_host()
        nbytes = 4 * n * A + 4 * n + 4 * n + 4 * n * S + 4 * n * S + 8 * (64 + 16)
        block = C.c_void_p()
        N.check(lib.nig_host_alloc(nbytes, C.byref(block)))
        buf = np.ctypeslib.as_array(C.cast(block, C.POINTER(C.c_uint8)), shape=(nbytes,))
        buf[:] = 0xA5
        off = [0]

        def carve(count, dtype):
            a = buf[off[0]:off[0] + count * np.dtype(dtype).itemsize].view(dtype)
            off[0] += count * np.dtype(dtype).itemsize + 64            # >= 64 canary bytes after every array ...
            off[0] = (off[0] + 15) // 16 * 16                          # ... and every array aligned like a C caller's would be
            return a
        act, rew, fl, vm = carve(n * A, np.float32), carve(n, np.float32), carve(n, np.uint8), carve(n, np.uint8)
        term, trunc = carve(n, np.uint8), carve(n, np.uint8)
        obs, nxt = carve(n * S, np.float32), carve(n * S, np.float32)
        act[:] = np.random.default_rng(0).uniform(-1, 1, n * A).astype(np.float32)
        io = N.StepIO()
        io.actions, io.reward, io.flags, io.viol_mask = act.ctypes.data, rew.ctypes.data, fl.ctypes.data, vm.ctypes.data
        io.terminated, io.truncated = term.ctypes.data, trunc.ctypes.data
        io.obs, io.next_obs = obs.ctypes.data, nxt.ctypes.data
        io.action_layout, io.aux_layout = N.LAYOUT_AOS, N.LAYOUT_AOS
        launches0 = env.launch_count
        for _ in range(3):
            N.check(lib.nig_step_host(env._h, C.byref(io)))
        assert env.launch_count - launches0 == 3                       # the zero-copy path: one launch per call, no staging kernels
        used = np.zeros(nbytes, bool)
        for a in (act, rew, fl, vm, term, trunc, obs, nxt):
            start = a.ctypes.data - buf.ctypes.data
            used[start:start + a.nbytes] = True
        assert (buf[~used] == 0xA5).all(), f"NIG_STEP_VEC={vec}: bytes outside the caller's arrays were overwritten"
        assert np.isfinite(rew).all() and (fl != 0xA5).all()
        assert np.array_equal(term, (fl & 1) != 0) and np.array_equal(trunc, (fl & 2) != 0), vec
        N.check(lib.nig_host_free(block))
        env.close()


def test_seeded_reset_is_reproducible(mods):
    """gym contract: reset(seed=s) twice gives the same first observation and the same noise afterwards (ADVICE r01)."""
    ni, N, O, torch = mods
    env = ni.make("ChemicalReactor-v0", device="cuda:0")
    o1, _ = env.reset(seed=42)
    t1 = [env.step(np.array([0.1, -0.2, 0.3], np.float32))[0].copy() for _ in range(5)]
    env.step(np.zeros(3, np.float32))
    o2, _ = env.reset(seed=42)
    t2 = [env.step(np.array([0.1, -0.2, 0.3], np.float32))[0].copy() for _ in range(5)]
    assert_bits_equal(o1, o2, "first observation")
    assert_bits_equal(np.stack(t1), np.stack(t2), "trajectory after the seeded reset")
    o3, _ = env.reset(seed=43)
    assert not np.array_equal(o1, o3)
    o4, _ = env.reset()                   # unseeded resets keep drawing fresh states
    assert not np.array_equal(o3, o4)
    env.close()
    venv = ni.TorchIndustrialEnv("ChemicalReactor-v0", 256, device="cuda:0", seed=1)
    a, _ = venv.reset(seed=7)
    a = a.clone()
    venv.step(torch.zeros((256, 3), device=venv.device))
    b, _ = venv.reset(seed=7)
    assert torch.equal(a, b)
    venv.close()


def test_allreduce_stats_through_the_c_abi_single_rank(mods):
    """nig_allreduce_stats with a communicator made by the C ABI's own helpers (ncclGetUniqueId / ncclCommInitRank through
    the dlopen()ed libnccl): on a one-rank communicator the grouped all-reduce (int64 SUM, fp64 SUM, extrema MAX) must leave
    the block unchanged. (World sizes > 1: tests/_nccl_worker.py under torchrun.)"""
    ni, N, O, torch = mods
    lib = N.lib()
    ident = (C.c_char * 128)()
    N.check(lib.nig_nccl_unique_id(C.cast(ident, C.c_void_p)))
    comm = C.c_void_p()
    N.check(lib.nig_nccl_comm_init(C.byref(comm), 1, C.cast(ident, C.c_void_p), 0, 0))
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, 4096, device=0, seed=3, max_episode_steps=30)
    env.reset_device()
    env.track_extrema(True)
    env.rollout_device(100, N.POLICY_UNIFORM)
    torch.cuda.synchronize()
    before_c, before_f = env.read_stats()
    before_x = env.read_extrema()
    st = int(torch.cuda.current_stream().cuda_stream)
    for _ in range(3):
        N.check(lib.nig_allreduce_stats(env._h, comm, st))
    torch.cuda.synchronize()
    after_c, after_f = env.read_stats()
    assert before_c.tolist() == after_c.tolist() and before_f.tolist() == after_f.tolist() and before_c[N.ST_EPISODES] > 0
    assert env.read_extrema() == before_x and before_x[0] is not None
    with pytest.raises(ValueError):
        N.check(lib.nig_allreduce_stats(env._h, None, st))
    N.check(lib.nig_nccl_comm_destroy(comm))
    env.close()


class _BangBang:
    """deterministic policy that ends reactor episodes at very different lengths (heats hard when cold)"""
    is_trained = True

    def predict(self, obs, deterministic=True):
        obs = np.atleast_2d(obs)
        a = np.zeros((obs.shape[0], 3), np.float32)
        a[:, 0] = np.where(obs[:, 0] < 321.0, 1.0, -0.2)
        return a


def test_batched_evaluation_uses_per_env_episode_quotas(mods):
    """evaluate_with_safety on a batched env runs, per env, a fixed quota of episodes to their end (utils.py:82-125 runs its
    n_episodes one after the other): exactly n_episodes are counted, env i contributes its FIRST quota_i episodes, and the
    result equals replaying those episodes one env at a time."""
    ni, N, O, torch = mods
    n, n_ep = 8, 21                                   # quotas 3,3,3,3,3,2,2,2
    env = ni.make("ChemicalReactor-v0", num_envs=n, seed=5, max_episode_steps=60)
    res = ni.evaluate_with_safety(_BangBang(), env, n_episodes=n_ep)
    env.close()
    # the same episodes, one env at a time (global env ids key the random streams, so env i alone reproduces shard i)
    rets, lens, viol = [], [], 0
    for i in range(n):
        e1 = ni.make("ChemicalReactor-v0", num_envs=1, batched=True, seed=5, max_episode_steps=60, env_id_offset=i)
        obs, _ = e1.reset()
        quota = n_ep // n + (1 if i < n_ep % n else 0)
        ep_r, ep_l = 0.0, 0
        while quota:
            obs, r, te, tr, info = e1.step(_BangBang().predict(obs))
            ep_r += float(r[0]); ep_l += 1
            viol += int(info["safety_metrics"].violation_count[0])
            if te[0] or tr[0]:
                rets.append(ep_r); lens.append(ep_l); ep_r, ep_l = 0.0, 0; quota -= 1
        e1.close()
    assert len(rets) == n_ep
    np.testing.assert_allclose(res["return_mean"], np.mean(rets), rtol=1e-12)
    np.testing.assert_allclose(res["length_mean"], np.mean(lens), rtol=1e-12)
    assert res["return_min"] == min(rets) and res["return_max"] == max(rets) and res["safety_violations"] == viol


def test_host_evaluated_constraints_vectorised_or_bounded(mods):
    """callable check_fns run on the host: a vectorised one costs one call per step; a per-env one is refused above
    HOSTMASK_LOOP_LIMIT envs instead of silently looping num_envs x constraints times in Python."""
    ni, N, O, torch = mods
    from neorl_industrial.core.types import SafetyConstraint
    n = 6000
    calls = []

    def hot(states, actions):
        calls.append(states.shape)
        return states[:, 0] <= 321.0

    env = ni.make("ChemicalReactor-v0", num_envs=n, seed=2)
    env.add_safety_constraint(SafetyConstraint("hot_vec", hot, -7.0, False, vectorized=True))
    obs, _ = env.reset()
    a = np.zeros((n, 3), np.float32)
    _, r1, _, _, info = env.step(a)
    assert calls == [(n, 12)]
    want = (obs[:, 0] > 321.0)
    assert np.array_equal((info["violation_mask"] >> 3) & 1, want.astype(np.uint8)) and want.any() and not want.all()
    env.add_safety_constraint(SafetyConstraint("hot_scalar", lambda s, a: s[0] <= 321.0, -7.0, False))
    with pytest.raises(ValueError, match="vectorised callable"):
        env.step(a)
    env.close()
    small = ni.make("ChemicalReactor-v0", num_envs=64, seed=2)
    small.add_safety_constraint(SafetyConstraint("hot_scalar", lambda s, a: s[0] <= 321.0, -7.0, False))
    o, _ = small.reset()
    _, _, _, _, info = small.step(np.zeros((64, 3), np.float32))
    assert np.array_equal((info["violation_mask"] >> 3) & 1, (o[:, 0] > 321.0).astype(np.uint8))
    small.close()


@pytest.mark.parametrize("bands", ["T", "P", "TP", "PT", "T_nan_hi"])
@pytest.mark.parametrize("extrema", [False, True])
def test_reactor_fast_loop_with_wrapper_bands(mods, bands, extrema):
    """BASELINE config 4: ChemicalReactor-v0 + SafetyWrapper temperature / pressure bands (non-critical, penalty on the
    PRE-step value, applied after the built-ins' penalties in constraint order). Such bounds ride along in the
    invariant-specialised loop (FastBounds); the population also holds warps that leave it (tripped e-stop, over-limit
    temperature, imminent truncation). 600 steps through nig_rollout_steps (env slices, K = 64) == the oracle bit for bit:
    states, episode words, per-constraint counters, per-env reward sums."""
    ni, N, O, torch = mods
    from neorl_industrial.vector import make_constraint
    f32 = lambda x: float(np.float32(x))
    spec = N.env_spec(N.ENV_CHEMICAL_REACTOR)
    builtins = [make_constraint(N.CON_BUILTIN, cid=k, penalty=spec.constraints[k].penalty, critical=bool(spec.constraints[k].critical))
                for k in range(3)]
    bT = make_constraint(N.CON_BOUND, si=0, lo=f32(305.0), hi=f32(325.0), penalty=-100.0)
    bP = make_constraint(N.CON_BOUND, si=1, lo=f32(101325.0), hi=f32(2.6e5), penalty=-37.5)
    bTn = make_constraint(N.CON_BOUND, si=0, lo=f32(305.0), hi=float("nan"), penalty=-3.0)       # always violated (a NaN bound compares false)
    cons = builtins + {"T": [bT], "P": [bP], "TP": [bT, bP], "PT": [bP, bT], "T_nan_hi": [bTn]}[bands]
    n = 6000 + 17
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=77, constraints=cons)
    ocons = [O.Con(c.kind, c.id, c.si, c.ai, c.coef, c.lo, c.hi, c.penalty, c.critical) for c in cons]
    orc = O.OracleEnv(O.REACTOR, n, auto_reset=True, seed=77, exp_mode=1, builtin=False, extra_cons=ocons)
    s0 = env.reset_host()
    assert_bits_equal(s0, orc.reset(), "reset")
    rng = np.random.default_rng(8)
    st = s0.copy()
    ep_step = np.zeros(n, np.int32)
    st[rng.choice(n, 30, replace=False), 8] = 1.0
    st[rng.choice(n, 30, replace=False), 0] = rng.uniform(349.0, 353.0, 30).astype(np.float32)
    ep_step[rng.choice(n, 300, replace=False)] = rng.integers(380, 500, 300)
    env.set_state_host(st, ep_step, np.zeros(n, np.int32), np.zeros(n, np.uint8))
    orc.state[:] = st
    orc.ep_step[:] = ep_step
    env.track_extrema(extrema)
    rsum = env.empty()
    env.rollout_device(70, N.POLICY_UNIFORM, reward_sum=rsum)
    o_rs = O.rollout(orc, 70, O.POLICY_UNIFORM, want_reward_sum=True)
    torch.cuda.synchronize()
    assert_bits_equal(rsum[:n].cpu().numpy(), o_rs, "reward sum with band penalties")
    env.rollout_steps_device(530, 64, N.POLICY_UNIFORM)
    O.rollout(orc, 530, O.POLICY_UNIFORM)
    torch.cuda.synchronize()
    st1, es, ev, dn = env.get_state_host()
    assert_bits_equal(st1, orc.state, "state"); assert_bits_equal(es, orc.ep_step, "ep_step"); assert_bits_equal(ev, orc.ep_viol, "ep_viol")
    c, _ = env.read_stats()
    assert c[:6].tolist() == orc.stats[:6].tolist()
    assert c[8:8 + len(cons)].tolist() == orc.stats[8:8 + len(cons)].tolist()
    assert c[8 + 3] > 0 and c[1] > 0                     # the first band fired; episodes ended (auto-resets inside the loop)
    env.close()


@pytest.mark.parametrize("use_tma", [True, False])
@pytest.mark.parametrize("extrema", [False, True])
def test_reactor_fast_loop_with_supplied_actions(mods, use_tma, extrema):
    """NIG_POLICY_ACTIONS takes the invariant-specialised loop too (actions staged by TMA boxes or read one step ahead into
    registers, np.clip in the draw, noise from the step's Philox block). Adversarial action tensors -- out of [-1, 1], NaN,
    +-inf, -0.0 -- and a population mixing warps inside / outside the invariants, several launches with horizons that are not
    multiples of the 16-step TMA box: everything == the oracle bit for bit (a NaN action fails the loop's guard and the step
    is redone by the generic loop, including the box hand-over of a CTA whose warps run different loops)."""
    ni, N, O, torch = mods
    n = 2048 + 300
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=13)
    orc = O.OracleEnv(O.REACTOR, n, seed=13, exp_mode=1)
    s0 = env.reset_host()
    assert_bits_equal(s0, orc.reset(), "reset")
    rng = np.random.default_rng(3)
    st = s0.copy()
    ep_step = np.zeros(n, np.int32)
    st[rng.choice(n, 20, replace=False), 8] = 1.0
    st[rng.choice(n, 20, replace=False), 0] = rng.uniform(349.0, 353.0, 20).astype(np.float32)
    st[32 * 7:32 * 8, 9] = 0.5                  # one whole warp outside the invariant
    ep_step[rng.choice(n, 150, replace=False)] = rng.integers(400, 500, 150)
    env.set_state_host(st, ep_step, np.zeros(n, np.int32), np.zeros(n, np.uint8))
    orc.state[:] = st
    orc.ep_step[:] = ep_step
    env.track_extrema(extrema)
    dev = env.torch_device()
    for K in (70, 16, 33, 1, 64):
        acts = rng.uniform(-1.4, 1.4, (K, n, env.A)).astype(np.float32)
        flat = acts.reshape(-1)
        k = flat.size
        flat[rng.choice(k, k // 400, replace=False)] = np.nan
        flat[rng.choice(k, k // 400, replace=False)] = np.inf
        flat[rng.choice(k, k // 400, replace=False)] = -np.inf
        flat[rng.choice(k, k // 200, replace=False)] = -0.0
        flat[rng.choice(k, k // 200, replace=False)] = 1.0
        d_act = torch.zeros((K, env.A, env.pitch), dtype=torch.float32, device=dev)
        d_act[:, :, :n] = torch.from_numpy(np.ascontiguousarray(acts.transpose(0, 2, 1))).to(dev)
        rsum = env.empty()
        env.rollout_device(K, N.POLICY_ACTIONS, actions=d_act, use_tma=use_tma, reward_sum=rsum)
        o_rs = np.zeros(n, np.float32)
        for t in range(K):
            _, r, _, _ = orc.step(acts[t], want_next_obs=False)
            o_rs = (o_rs + r).astype(np.float32)
        torch.cuda.synchronize()
        _compare(env, orc, N, f"after a {K}-step launch of supplied actions")
        assert_bits_equal(rsum[:n].cpu().numpy(), o_rs, "per-env reward sum")
    env.close()


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_rollout_steps_graph_replay_equals_plain_enqueue(mods, monkeypatch, name):
    """nig_rollout_steps replays its sliced launch sequence from a captured CUDA graph once a call pattern repeats (first call:
    plain enqueue, second: capture + replay, later: replay; a different horizon in between re-arms the capture). Same calls on
    a handle created with NIG_STEPS_GRAPH=0: bit-identical states, episode words, per-env sums and counters."""
    ni, N, O, torch = mods
    kind = KINDS[name]
    n = 40_000 + 5
    res = []
    for graph in ("1", "0"):
        monkeypatch.setenv("NIG_STEPS_GRAPH", graph)
        env = ni.NativeEnv(kind, n, device=0, seed=17)
        env.reset_device()
        rsum = env.empty()
        launches0 = env.launch_count
        for horizon in (150, 150, 150, 150, 70, 150, 150):
            env.rollout_steps_device(horizon, 64, N.POLICY_UNIFORM, reward_sum=rsum)
        torch.cuda.synchronize()
        st, es, ev, dn = env.get_state_host()
        c, _ = env.read_stats()
        res.append((st, es, ev, dn, rsum[:n].cpu().numpy(), c.copy(), env.tick, env.launch_count - launches0))
        env.close()
    g, p = res
    assert_bits_equal(g[0], p[0], "state"); assert_bits_equal(g[1], p[1], "ep_step"); assert_bits_equal(g[2], p[2], "ep_viol")
    assert_bits_equal(g[4], p[4], "per-env reward sum of the last call")
    assert g[5].tolist() == p[5].tolist()
    assert g[6] == p[6] == 5 * 150 + 70 + 150
    assert g[7] == p[7] + 5            # calls 2, 3, 4, 6, 7 are replays, each with its tick-setting kernel


@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_step_without_device_counters(mods, name):
    """nig_track_step_stats(env, 0): single steps skip the device counter block (IndustrialEnv.step has none) -- states, rewards,
    flags, violation masks and episode words are those of a counting handle bit for bit, the counters stay where they were,
    and the fused rollout keeps counting."""
    ni, N, O, torch = mods
    kind = KINDS[name]
    n = 70_000 + 3                                     # above the persistent-pipeline threshold of none, below for all: both kernels appear across envs
    envs = [ni.NativeEnv(kind, n, device=0, seed=23) for _ in range(2)]
    quiet, counting = envs
    quiet.track_step_stats(False)
    for e in envs:
        e.reset_device()
    dev = quiet.torch_device()
    torch.manual_seed(0)
    outs = []
    for e in envs:
        rew, fl, vm = e.empty(), e.empty(dtype=torch.uint8), e.empty(dtype=torch.uint8)
        g = torch.Generator(device=dev); g.manual_seed(5)
        for _ in range(40):
            acts = torch.rand((e.A, e.pitch), device=dev, generator=g) * 2.6 - 1.3
            e.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
        torch.cuda.synchronize()
        outs.append((rew[:n].cpu().numpy(), fl[:n].cpu().numpy(), vm[:n].cpu().numpy()))
    sq, sc = quiet.get_state_host(), counting.get_state_host()
    assert_bits_equal(sq[0], sc[0], "state"); assert_bits_equal(sq[1], sc[1], "ep_step"); assert_bits_equal(sq[2], sc[2], "ep_viol")
    assert_bits_equal(outs[0][0], outs[1][0], "reward of the last step")
    assert np.array_equal(outs[0][1], outs[1][1]) and np.array_equal(outs[0][2], outs[1][2])
    cq, _ = quiet.read_stats()
    cc, _ = counting.read_stats()
    assert cq[N.ST_STEPS] == 0 and cc[N.ST_STEPS] == 40 * n
    quiet.rollout_device(16, N.POLICY_UNIFORM)
    torch.cuda.synchronize()
    cq, _ = quiet.read_stats()
    assert cq[N.ST_STEPS] == 16 * n
    for e in envs:
        e.close()
