"""Generate the golden fixtures by running the UNMODIFIED reference env code (teacher-forced).

Run in the build container only (needs /root/reference):  python tests/golden/make_golden.py
Reference version: _version.py -> 0.1.dev68+g9b77c89e2.d20250827; numpy 2.3.5 (NEP 50), fp32 actions,
fp32-representable noise (SURVEY.md section 8c "canonical for parity").

Fixtures (all small, committed; a set larger than 1 MB is stored as parts <name>.1.npz, <name>.2.npz, ... that
tests/util.py:load_golden merges):
  <env>_forced.npz : M independent (state, ep_step, action, noise) -> env.step() tuples, sampled to hit every
                     branch of the dynamics / reward / constraint / termination logic.
  <env>_trace.npz  : BASELINE config #1 -- one env, 1000 steps, random fp32 actions, reset on done; everything
                     needed to replay it teacher-forced (states, actions, noise, reset states, outputs).
  reactor_freerun.npz : 16 free-running 500-step episodes (actions + noise recorded) for the drift test.
  <env>_dataset_stats.json : summary statistics of the reference's get_dataset(quality) for every quality.
  policy_forced.npz : get_dataset's POLICY, teacher-forced -- per env x quality ~2000 transitions of the reference's own
                     get_dataset run: the observation the policy saw, every random value it drew (coin, normals,
                     uniforms; recorded by interposing np.random.*), and the action it stored.
  baseline_agents.npz : benchmarks/baseline_agents.py (loaded by file path, pure numpy) driven over state sequences:
                     PID (integral / derivative state), MPC heuristic, Constant -> float64 actions.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
import ref_loader  # noqa: E402
from util import save_golden  # noqa: E402

ENV_CLASS = {"reactor": "ChemicalReactorEnv", "grid": "PowerGridEnv", "robot": "RobotAssemblyEnv"}
NOISE_SHAPES = {"reactor": [None, None], "grid": [8, 8, 7], "robot": []}
NOISE_SIGMA = {"reactor": [0.1, 500.0], "grid": [0.005, 1.0, 2.0], "robot": []}
NZ = {"reactor": 2, "grid": 23, "robot": 0}


def draw_noise(rng, name):
    """fp32-representable noise, flat [NZ], plus the list to push into the NoiseQueue."""
    parts, flat = [], []
    for shape, sig in zip(NOISE_SHAPES[name], NOISE_SIGMA[name]):
        if shape is None:
            v = np.float32(rng.normal(0, sig))
            parts.append(float(v)); flat.append(np.array([v], np.float32))
        else:
            v = rng.normal(0, sig, shape).astype(np.float32)
            parts.append(v.astype(np.float64)); flat.append(v)
    return parts, (np.concatenate(flat) if flat else np.zeros(0, np.float32))


def forced_step(env, q, state, ep_step, action, noise_parts):
    env.state = state.copy()
    env.current_step = int(ep_step)
    env.done = False
    env.violation_count = 0
    env.total_violations = 0
    q.queue.clear()
    q.push(*noise_parts)
    obs, reward, terminated, truncated, info = env.step(action.copy())
    sm = info["safety_metrics"]
    assert not q.queue
    return (obs.astype(np.float32), np.float64(reward), bool(terminated), bool(truncated),
            int(sm.violation_count), int(sm.critical_violations), bool(info["critical_shutdown"]),
            int(info["violations"]))


def viol_mask_of(env, state, action):
    a = np.clip(action, env.action_space.low, env.action_space.high)
    m = 0
    for k, c in enumerate(env.safety_constraints):
        if not c.check_fn(state, a):
            m |= 1 << k
    return m


# ------------------------------------------------------------------------------------------------
def sample_reactor_states(rng, env, m):
    S = np.zeros((m, 12), np.float32)
    steps = np.zeros(m, np.int32)
    for i in range(m):
        mode = i % 4
        if mode == 0:      # nominal: reset distribution
            S[i] = env._get_initial_state()
            steps[i] = rng.integers(0, 499)
        else:              # wide: every branch reachable
            S[i] = [rng.uniform(300, 360), rng.uniform(2.0e5, 5.3e5), rng.uniform(8, 102), rng.uniform(4, 52),
                    rng.uniform(0, 2) if rng.random() < 0.9 else 0.0, rng.uniform(49.9, 100), rng.uniform(285, 300),
                    0.0 if rng.random() < 0.5 else rng.uniform(0, 100), float(rng.random() < 0.3),
                    float(rng.random() < 0.4), rng.uniform(0, 100), rng.uniform(0, 51)]
            steps[i] = rng.choice([rng.integers(0, 497), 498, 499]) if mode == 3 else rng.integers(0, 499)
        if mode == 2:      # clamp edges hit exactly
            j = i % 12
            if j == 2: S[i, 3] = 5.0
            if j == 6: S[i, 3] = 50.0
            if j == 10: S[i, 2] = 10.0 if rng.random() < 0.5 else 100.0
            if i % 5 == 0: S[i, 10] = rng.choice([0.0, 100.0, 4.99, 95.01, 20.0, 90.0, 30.0, 80.0])
            if i % 7 == 0: S[i, 0] = rng.choice([350.0, 345.0, 340.0, 349.99, 350.01])
            if i % 11 == 0: S[i, 1] = rng.choice([506625.0, 480000.0, 506625.03, 101325.0])
    return S, steps


def sample_grid_states(rng, env, m):
    S = np.zeros((m, 32), np.float32)
    steps = np.zeros(m, np.int32)
    for i in range(m):
        S[i] = env._get_initial_state()
        mode = i % 4
        steps[i] = rng.integers(0, 999)
        if mode >= 1:
            S[i, 0] = rng.uniform(-1.2, 1.2) if mode == 1 else rng.normal(0, 0.3)
        if mode == 2:
            S[i, 1:9] = rng.uniform(0.88, 1.12, 8)
            S[i, 9:17] = rng.uniform(-1, 101, 8)
        if mode == 3:
            steps[i] = rng.choice([998, 999, rng.integers(0, 998)])
            k = rng.integers(0, 8)
            S[i, 1 + k] = rng.choice([0.95, 1.05, 0.9, 1.1, 0.94999, 1.05001])
            S[i, 9 + k] = rng.choice([0.0, 100.0, 99.5, 0.5])
            S[i, 17:25] = np.maximum(S[i, 17:25] + rng.normal(0, 30, 8), 0)
    return S, steps


def sample_robot_states(rng, env, m):
    S = np.zeros((m, 24), np.float32)
    steps = np.zeros(m, np.int32)
    for i in range(m):
        mode = i % 4
        steps[i] = rng.integers(0, 999) if mode != 3 else rng.choice([998, 999, 5])
        if mode == 0:
            S[i] = env._get_initial_state()
        else:
            q = rng.uniform(-np.pi, np.pi, 7) if mode == 1 else rng.uniform(-1.0, 1.0, 7)
            if mode == 2 and i % 8 == 2:
                # near the assembly target: search a configuration close to [0.3, 0, 0.4]
                best = None
                for _ in range(4000):
                    qq = rng.uniform(-np.pi, np.pi, 7)
                    p, _ = env._forward_kinematics(qq)
                    d = np.linalg.norm(p - env.target_position)
                    if best is None or d < best[0]:
                        best = (d, qq)
                q = best[1]
            if i % 9 == 0:
                q[rng.integers(0, 7)] = rng.choice([np.pi, -np.pi, 2.0, -2.0, 1.99, 3.1])
            p, quat = env._forward_kinematics(q)
            S[i, 0:3] = p + (rng.normal(0, 0.02, 3) if mode == 1 else 0)
            S[i, 3:7] = quat
            S[i, 7:14] = q
            S[i, 14:17] = rng.normal(0, 0.5, 3)
            if i % 6 == 0:
                S[i, 18:21] = rng.choice([0.0, 10.0, 49.9, 50.0, 79.0, 81.0, -60.0], 3)
            S[i, 21:24] = rng.uniform(0, 1, 3)
    return S, steps


SAMPLERS = {"reactor": sample_reactor_states, "grid": sample_grid_states, "robot": sample_robot_states}


def make_forced(envs, name, m, seed):
    rng = np.random.default_rng(seed)
    np.random.seed(seed)
    env = getattr(envs, ENV_CLASS[name])()
    S, steps = SAMPLERS[name](rng, env, m)
    A = rng.uniform(-1.5, 1.5, (m, env.action_dim)).astype(np.float32)
    A[::13] = np.clip(A[::13], -1, 1)
    A[5::17] = 0.0
    out = {k: [] for k in ("next_state", "reward", "terminated", "truncated", "n_viol", "n_crit", "crit", "viol_mask", "noise")}
    with ref_loader.NoiseQueue() as q:
        for i in range(m):
            parts, flat = draw_noise(rng, name)
            vm = viol_mask_of(env, S[i], A[i])
            ns, r, te, tr, nv, nc, cs, ev = forced_step(env, q, S[i], steps[i], A[i], parts)
            assert ev == nv and bin(vm).count("1") == nv
            for k, v in zip(("next_state", "reward", "terminated", "truncated", "n_viol", "n_crit", "crit", "viol_mask", "noise"),
                            (ns, r, te, tr, nv, nc, cs, vm, flat)):
                out[k].append(v)
    save_golden(os.path.join(HERE, f"{name}_forced"),
                state=S, ep_step=steps, action=A,
                noise=np.array(out["noise"], np.float32).reshape(m, NZ[name]),
                next_state=np.array(out["next_state"], np.float32),
                reward=np.array(out["reward"], np.float64),
                terminated=np.array(out["terminated"], bool), truncated=np.array(out["truncated"], bool),
                n_viol=np.array(out["n_viol"], np.int32), n_crit=np.array(out["n_crit"], np.int32),
                crit=np.array(out["crit"], bool), viol_mask=np.array(out["viol_mask"], np.uint8))
    te, tr, cr = np.array(out["terminated"]), np.array(out["truncated"]), np.array(out["crit"])
    print(f"{name}_forced: {m} tuples, terminated {te.sum()}, truncated {tr.sum()}, critical {cr.sum()}, "
          f"violations {np.sum(out['n_viol'])}")


def make_trace(envs, name, n_steps, seed):
    """BASELINE config #1: performance_benchmark.py:106-133 loop, recorded for teacher-forced replay."""
    rng = np.random.default_rng(seed)
    np.random.seed(seed)
    env = getattr(envs, ENV_CLASS[name])()
    env.action_space.seed(seed)
    obs, _ = env.reset()
    rec = {k: [] for k in ("state", "action", "noise", "next_state", "reward", "terminated", "truncated", "n_viol",
                           "crit", "viol_mask", "ep_step", "reset_state", "ep_violations", "total_violations")}
    with ref_loader.NoiseQueue() as q:
        for t in range(n_steps):
            a = env.action_space.sample()
            parts, flat = draw_noise(rng, name)
            q.queue.clear(); q.push(*parts)
            s0 = env.state.copy(); st0 = env.current_step
            vm = viol_mask_of(env, s0, a)
            obs, r, te, tr, info = env.step(a)
            rec["state"].append(s0); rec["action"].append(a); rec["noise"].append(flat)
            rec["next_state"].append(obs.copy()); rec["reward"].append(np.float64(r))
            rec["terminated"].append(te); rec["truncated"].append(tr)
            rec["n_viol"].append(info["safety_metrics"].violation_count); rec["crit"].append(info["critical_shutdown"])
            rec["viol_mask"].append(vm); rec["ep_step"].append(st0)
            rec["ep_violations"].append(info["violations"]); rec["total_violations"].append(info["total_violations"])
            if te or tr:
                np.random.normal = q._orig          # reset draws come from the real global RNG
                obs, _ = env.reset()
                np.random.normal = q._normal
                rec["reset_state"].append(env.state.copy())
            else:
                rec["reset_state"].append(np.zeros(env.state_dim, np.float32))
    np.savez_compressed(os.path.join(HERE, f"{name}_trace.npz"),
                        state=np.array(rec["state"], np.float32), action=np.array(rec["action"], np.float32),
                        noise=np.array(rec["noise"], np.float32).reshape(n_steps, NZ[name]),
                        next_state=np.array(rec["next_state"], np.float32), reward=np.array(rec["reward"], np.float64),
                        terminated=np.array(rec["terminated"], bool), truncated=np.array(rec["truncated"], bool),
                        n_viol=np.array(rec["n_viol"], np.int32), crit=np.array(rec["crit"], bool),
                        viol_mask=np.array(rec["viol_mask"], np.uint8), ep_step=np.array(rec["ep_step"], np.int32),
                        reset_state=np.array(rec["reset_state"], np.float32),
                        ep_violations=np.array(rec["ep_violations"], np.int32),
                        total_violations=np.array(rec["total_violations"], np.int32))
    d = np.array(rec["terminated"]) | np.array(rec["truncated"])
    print(f"{name}_trace: {n_steps} steps, {d.sum()} episodes ended, {np.sum(rec['n_viol'])} violations")


def make_freerun(envs, n_ep, seed):
    rng = np.random.default_rng(seed)
    np.random.seed(seed)
    env = envs.ChemicalReactorEnv()
    T = 500
    init = np.zeros((n_ep, 12), np.float32)
    A = rng.uniform(-1, 1, (n_ep, T, 3)).astype(np.float32)
    A[n_ep // 2:] *= 0.3      # gentler actions -> longer episodes
    NZv = np.zeros((n_ep, T, 2), np.float32)
    states = np.zeros((n_ep, T, 12), np.float32)
    rewards = np.zeros((n_ep, T), np.float64)
    flags = np.zeros((n_ep, T), np.uint8)
    length = np.zeros(n_ep, np.int32)
    with ref_loader.NoiseQueue() as q:
        for e in range(n_ep):
            np.random.normal = q._orig
            env.reset()
            np.random.normal = q._normal
            init[e] = env.state
            for t in range(T):
                parts, flat = draw_noise(rng, "reactor")
                NZv[e, t] = flat
                q.queue.clear(); q.push(*parts)
                obs, r, te, tr, info = env.step(A[e, t])
                states[e, t] = obs; rewards[e, t] = r
                flags[e, t] = (1 if te else 0) | (2 if tr else 0) | (4 if info["critical_shutdown"] else 0)
                length[e] = t + 1
                if te or tr:
                    break
    np.savez_compressed(os.path.join(HERE, "reactor_freerun.npz"), init=init, action=A, noise=NZv,
                        states=states, rewards=rewards, flags=flags, length=length)
    print("reactor_freerun: lengths", length.tolist())


class PolicyRecorder:
    """Pass-through interposer on np.random.normal / uniform / random / rand that records, per transition of a running
    get_dataset, the draws made by the POLICY (those outside env.reset / env.step) and the action handed to env.step."""

    def __init__(self, env):
        self.env, self.in_env, self.pending, self.rows = env, 0, [], []
        self._orig = {k: getattr(np.random, k) for k in ("normal", "uniform", "random", "rand")}
        self._step, self._reset = env.step, env.reset

    def _wrap_draw(self, name):
        orig = self._orig[name]

        def f(*a, **kw):
            v = orig(*a, **kw)
            if not self.in_env:
                self.pending.append((name, a, np.array(v, np.float64).copy()))
            return v
        return f

    def __enter__(self):
        for k in self._orig:
            setattr(np.random, k, self._wrap_draw(k))

        def step(action):
            self.rows.append((self.env.state.copy(), self.pending, np.array(action, np.float64).copy()))
            self.pending = []
            self.in_env += 1
            try:
                return self._step(action)
            finally:
                self.in_env -= 1

        def reset(*a, **kw):
            assert not self.pending
            self.in_env += 1
            try:
                return self._reset(*a, **kw)
            finally:
                self.in_env -= 1
        self.env.step, self.env.reset = step, reset
        return self

    def __exit__(self, *exc):
        for k, v in self._orig.items():
            setattr(np.random, k, v)
        del self.env.step, self.env.reset
        return False


def forced_inputs(name, draws):
    """Recorded np.random calls of one transition -> (coin, z[8] = normal / scale, u[8] = uniform mapped to [-1, 1])."""
    coin, z, u = np.nan, np.zeros(8), np.zeros(8)
    nz = nu = 0
    for fn, args, v in draws:
        if fn in ("random", "rand"):
            assert np.isnan(coin) and v.ndim == 0
            coin = float(v)
        elif fn == "normal":
            assert args[0] == 0 and v.ndim == 0
            z[nz] = float(v) / args[1]; nz += 1
        else:
            lo, hi = float(args[0]), float(args[1])
            assert lo == -hi
            for x in np.atleast_1d(v):
                u[nu] = x / hi; nu += 1
    return coin, z, u


def make_policy_forced(envs, seed, per_case=2000):
    rng = np.random.default_rng(seed)
    out = {}
    for name in ("reactor", "grid", "robot"):
        for quality in ("expert", "medium", "mixed", "random"):
            np.random.seed(seed)
            env = getattr(envs, ENV_CLASS[name])()
            with PolicyRecorder(env) as rec:
                d = env.get_dataset(quality)
            rows = rec.rows
            assert len(rows) == len(d["actions"])
            stored = d["actions"]
            for i in rng.choice(len(rows), 50, replace=False):    # the recorder sees what the dataset stores
                assert np.array_equal(np.asarray(rows[i][2], np.float32), stored[i]), (name, quality, i)
                assert np.array_equal(rows[i][0], d["observations"][i])
            pick = np.sort(rng.choice(len(rows), min(per_case, len(rows)), replace=False))
            obs = np.array([rows[i][0] for i in pick], np.float32)
            fi = [forced_inputs(name, rows[i][1]) for i in pick]
            key = f"{name}_{quality}"
            out[key + "_obs"] = obs
            out[key + "_coin"] = np.array([f[0] for f in fi], np.float64)
            out[key + "_z"] = np.array([f[1] for f in fi], np.float32)
            out[key + "_u"] = np.array([f[2] for f in fi], np.float32)
            out[key + "_action"] = stored[pick].astype(np.float32)
            c = out[key + "_coin"]
            print(f"policy_forced {key}: {len(rows)} transitions recorded, {len(pick)} kept, coin drawn in "
                  f"{np.isfinite(c).sum()}, normals in {(np.abs(out[key + '_z']).sum(1) > 0).sum()}, "
                  f"uniforms in {(np.abs(out[key + '_u']).sum(1) > 0).sum()}")
    save_golden(os.path.join(HERE, "policy_forced"), **out)


def make_baseline_goldens(seed):
    """benchmarks/baseline_agents.py:28-114, imported by file path (pure numpy)."""
    import importlib.util
    path = os.path.join(ref_loader.REFERENCE_SRC, "neorl_industrial", "benchmarks", "baseline_agents.py")
    spec = importlib.util.spec_from_file_location("_ref_baseline_agents", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    rng = np.random.default_rng(seed)
    out = {}
    T, n = 64, 48
    for name, (S, A) in {"reactor": (12, 3), "grid": (32, 8), "robot": (24, 7)}.items():
        tr = np.load(os.path.join(HERE, f"{name}_trace.npz"))["state"]
        # n independent agents, each fed T consecutive states of the reference trace from a different offset,
        # plus (last quarter) states scaled so that the clip at +-1 and the integral wind-up are both exercised
        starts = rng.integers(0, len(tr) - T, n)
        states = np.stack([tr[s0:s0 + T] for s0 in starts], 1).astype(np.float32)      # [T, n, S]
        states[:, 3 * n // 4:, :A] *= 0.01
        # setpoint near the mean of the process variables and gains scaled by their spread: O(1) actions, partly clipped
        setpoint = tr[:, :A].astype(np.float64).mean(0) + rng.normal(0, 0.05, A)
        spread = float(tr[:, :A].astype(np.float64).std(0).max()) + 1e-3
        gains = np.array([0.8, 0.05, 0.02]) / spread
        const = rng.uniform(-1, 1, A)
        out[f"{name}_pid_gains"] = gains
        cases = {
            "pid": lambda: mod.PIDControllerAgent(S, A, kp=gains[0], ki=gains[1], kd=gains[2], setpoint=setpoint.copy()),
            "pid_default": lambda: mod.PIDControllerAgent(S, A),
            "mpc": lambda: mod.MPC_Agent(S, A),
            "constant": lambda: mod.ConstantAgent(S, A, constant_action=const.copy()),
        }
        out[f"{name}_states"] = states
        out[f"{name}_setpoint"] = setpoint
        out[f"{name}_constant"] = const
        for cname, mk in cases.items():
            acts = np.zeros((T, n, A), np.float64)
            for i in range(n):
                agent = mk()
                for t in range(T):
                    acts[t, i] = agent.act(states[t, i])
            out[f"{name}_{cname}_actions"] = acts
        print(f"baseline_agents {name}: {T} x {n} states, |pid action| == 1 in "
              f"{np.mean(np.abs(out[f'{name}_pid_actions']) == 1.0):.2f} of the entries")
    # the factory and the random agent's range (distribution only: it draws from the global numpy stream)
    np.random.seed(seed)
    ra = mod.BaselineAgentFactory.create("random", 12, 3, action_low=-0.5, action_high=0.25)
    draws = np.array([ra.act(np.zeros(12)) for _ in range(4000)])
    out["random_low_high_mean_std"] = np.array([draws.min(), draws.max(), draws.mean(), draws.std()])
    np.savez_compressed(os.path.join(HERE, "baseline_agents.npz"), **out)


def make_dataset_stats(envs, seed, name="reactor"):
    out = {}
    for quality in ("mixed", "expert", "medium", "random"):
        np.random.seed(seed)
        env = getattr(envs, ENV_CLASS[name])()
        d = env.get_dataset(quality)
        term = d["terminals"]
        ends = np.flatnonzero(term)
        out[quality] = {
            "n": int(len(d["rewards"])), "n_terminals": int(term.sum()),
            "obs_dtype": str(d["observations"].dtype), "act_dtype": str(d["actions"].dtype),
            "rew_dtype": str(d["rewards"].dtype), "term_dtype": str(d["terminals"].dtype),
            "keys": sorted(d.keys()),
            "reward_mean": float(d["rewards"].mean()), "reward_std": float(d["rewards"].std()),
            "reward_median": float(np.median(d["rewards"])),
            "action_mean": d["actions"].mean(0).tolist(), "action_std": d["actions"].std(0).tolist(),
            "obs_mean": d["observations"].mean(0).tolist(), "obs_std": d["observations"].std(0).tolist(),
            "frac_action_saturated": float(np.mean(np.abs(d["actions"]) >= 1.0)),
            "timeouts_any": bool(d["timeouts"].any()) if "timeouts" in d else False,
            "episode_len_mean": float(len(term) / max(1, int(term.sum()))) if name != "reactor" else None,
        }
        print(quality, {k: out[quality][k] for k in ("n", "n_terminals", "reward_mean", "reward_std")})
    with open(os.path.join(HERE, f"{name}_dataset_stats.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    envs = ref_loader.load_reference_envs()
    which = sys.argv[1:] or ["forced", "trace", "freerun", "dataset", "dataset_all", "policy", "baselines"]
    if "forced" in which:
        make_forced(envs, "reactor", 6000, 1)
        make_forced(envs, "grid", 3000, 2)
        make_forced(envs, "robot", 2000, 3)
    if "trace" in which:
        make_trace(envs, "reactor", 1000, 0)
        make_trace(envs, "grid", 1000, 0)
        make_trace(envs, "robot", 1000, 0)
    if "freerun" in which:
        make_freerun(envs, 16, 5)
    if "dataset" in which:
        make_dataset_stats(envs, 0)
    if "dataset_all" in which:
        make_dataset_stats(envs, 0, "grid")
        make_dataset_stats(envs, 0, "robot")
    if "policy" in which:
        make_policy_forced(envs, 11)
    if "baselines" in which:
        make_baseline_goldens(12)
