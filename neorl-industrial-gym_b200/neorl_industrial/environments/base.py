"""``IndustrialEnv``: the reference's gym-style env API (environments/base.py:19-228) over the CUDA path.

One object drives ``num_envs`` independent envs resident on one B200. With ``num_envs == 1`` (the
default, = ``ni.make(env_id)`` upstream) ``reset``/``step`` return exactly the reference's shapes and
types -- obs ``float32[S]``, scalar reward, Python bools, ``info`` with the same keys -- and ``step``
after done raises ``RuntimeError`` like base.py:159-160. With ``num_envs > 1`` the same calls are
batched: arrays with a leading env axis, ``auto_reset=True`` by default.

All arithmetic (clip, constraints, dynamics, reward, penalties, termination, reset draws) runs in the
sm_100a kernels; this class only marshals arguments and builds ``info``. There is no CPU code path.
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, Tuple

import numpy as np

from .. import _native as N
from ..core.types import BatchedSafetyMetrics, SafetyConstraint, SafetyMetrics
from ..rollouts import resolve_policy
from ..spaces import Box
from ..vector import NativeEnv, make_constraint


class IndustrialEnv:
    ENV_ID: str = ""
    ENV_KIND: int = -1
    REWARD_IS_FLOAT32 = False     # reactor rewards are np.float32 upstream, grid/robot Python floats (SURVEY App. E.6)
    metadata: Dict[str, Any] = {"render_modes": []}

    def __init__(self, state_dim: int, action_dim: int, safety_constraints: Optional[List[SafetyConstraint]] = None,
                 max_episode_steps: int = 1000, dt: float = 0.1, *, num_envs: int = 1, device="cuda",
                 seed: Optional[int] = None, auto_reset: Optional[bool] = None, env_id_offset: int = 0,
                 batched: Optional[bool] = None, copy: bool = True):
        self.state_dim = state_dim
        self.action_dim = action_dim
        self.max_episode_steps = max_episode_steps
        self.dt = dt
        self.num_envs = int(num_envs)
        self.batched = bool(batched) if batched is not None else self.num_envs > 1
        self.auto_reset = bool(auto_reset) if auto_reset is not None else self.batched
        self.copy = copy
        self.safety_constraints: List[SafetyConstraint] = list(safety_constraints or [])
        self.info: Dict[str, Any] = {}
        self.observation_space = Box(-np.inf, np.inf, (state_dim,), np.float32)
        self.action_space = Box(-1.0, 1.0, (action_dim,), np.float32, seed=seed)
        self.np_random = np.random.default_rng(seed)
        self._seed = 0 if seed is None else int(seed)
        self.native = NativeEnv(self.ENV_KIND, self.num_envs, device=device, seed=self._seed, auto_reset=self.auto_reset,
                                max_episode_steps=max_episode_steps, env_id_offset=env_id_offset,
                                constraints=self._native_constraints())
        assert self.native.S == state_dim and self.native.A == action_dim
        # host mirrors (refreshed from every reset/step output; never used for arithmetic)
        self._state = None
        self._ep_step = np.zeros(self.num_envs, np.int64)
        self._ep_viol = np.zeros(self.num_envs, np.int64)
        self._done = np.zeros(self.num_envs, bool)
        self._total_violations_base = 0

    # ------------------------------------------------------------------ constraints
    def _native_constraints(self):
        out, bit = [], 0
        for c in self.safety_constraints:
            nat = getattr(c, "_native", None)
            if nat is None:
                if bit > 7:
                    raise ValueError("at most 8 host-evaluated (callable) constraints are supported")
                out.append(make_constraint(N.CON_HOSTMASK, cid=bit, penalty=c.penalty, critical=c.critical))
                bit += 1
            elif nat[0] == "builtin":
                out.append(make_constraint(N.CON_BUILTIN, cid=nat[1], penalty=c.penalty, critical=c.critical))
            elif nat[0] == "bound":
                _, si, ai, coef, lo, hi = nat
                out.append(make_constraint(N.CON_BOUND, si=si, ai=ai, coef=coef, lo=lo, hi=hi, penalty=c.penalty,
                                           critical=c.critical))
            else:
                raise ValueError(f"unknown native constraint descriptor {nat!r}")
        if len(out) > N.MAX_CONSTRAINTS:
            raise ValueError(f"at most {N.MAX_CONSTRAINTS} safety constraints are supported (got {len(out)})")
        return out

    def _host_constraints(self):
        return [c for c in self.safety_constraints if getattr(c, "_native", None) is None]

    def add_safety_constraint(self, constraint: SafetyConstraint) -> None:
        """base.py:220-222"""
        self.safety_constraints.append(constraint)
        try:
            self.native.set_constraints(self._native_constraints())
        except Exception:
            self.safety_constraints.pop()
            raise

    def remove_safety_constraint(self, name: str) -> None:
        """base.py:224-228"""
        self.safety_constraints = [c for c in self.safety_constraints if c.name != name]
        self.native.set_constraints(self._native_constraints())

    # callable check_fns are evaluated on the host, one Python call per env and constraint and step: fine for the single-env
    # gym API, hopeless for a large batch -- above this many envs only vectorised callables (SafetyConstraint(...,
    # vectorized=True): check_fn(states [n, S], actions [n, A]) -> bool [n]) or declarative BoundConstraints are accepted
    HOSTMASK_LOOP_LIMIT = 4096

    def _hostmask(self, actions: np.ndarray) -> Optional[np.ndarray]:
        host = self._host_constraints()
        if not host:
            return None
        a = np.clip(actions, self.action_space.low, self.action_space.high)
        n = self.num_envs
        mask = np.zeros(n, np.uint8)
        for bit, c in enumerate(host):
            if getattr(c, "vectorized", False):
                try:
                    ok = np.asarray(c.check_fn(self._state, a)).astype(bool).reshape(n)
                except Exception:          # base.py:109-113: an exception counts as a violation
                    ok = np.zeros(n, bool)
            else:
                if n > self.HOSTMASK_LOOP_LIMIT:
                    raise ValueError(
                        f"constraint {c.name!r} is a Python callable evaluated per env on the host ({n} envs x every step); "
                        f"above {self.HOSTMASK_LOOP_LIMIT} envs use safety.BoundConstraint (evaluated in-kernel) or a "
                        "vectorised callable: SafetyConstraint(..., vectorized=True)")
                ok = np.ones(n, bool)
                for i in range(n):
                    try:
                        ok[i] = bool(c.check_fn(self._state[i], a[i]))
                    except Exception:
                        ok[i] = False
            mask[~ok] |= np.uint8(1 << bit)
        return mask

    # ------------------------------------------------------------------ reference attributes
    # num_envs == 1: host mirrors are kept eagerly (reference semantics, cheap). Batched: nothing is
    # mirrored per step; the properties read the device state on demand.
    def _pull(self):
        s, st, vi, dn = self.native.get_state_host()
        self._state, self._ep_step, self._ep_viol, self._done = s, st.astype(np.int64), vi.astype(np.int64), dn

    @property
    def state(self):
        if self._state is None:
            return None
        if self.batched:
            self._pull()
            return self._state
        return self._state[0]

    @state.setter
    def state(self, value):
        """Teacher forcing / checkpoint restore: overwrite the device state."""
        s = np.ascontiguousarray(value, np.float32).reshape(self.num_envs, self.state_dim)
        self.native.set_state_host(state=s)
        self._state = s.copy()

    @property
    def current_step(self):
        if self.batched:
            self._pull()
            return self._ep_step
        return int(self._ep_step[0])

    @current_step.setter
    def current_step(self, value):
        st = np.broadcast_to(np.asarray(value, np.int32), (self.num_envs,)).copy()
        self.native.set_state_host(ep_step=st)
        self._ep_step = st.astype(np.int64)

    @property
    def violation_count(self):
        if self.batched:
            self._pull()
            return self._ep_viol
        return int(self._ep_viol[0])

    @violation_count.setter
    def violation_count(self, value):
        v = np.broadcast_to(np.asarray(value, np.int32), (self.num_envs,)).copy()
        self.native.set_state_host(ep_viol=v)
        self._ep_viol = v.astype(np.int64)

    @property
    def done(self):
        if self.batched:
            self._pull()
            return self._done
        return bool(self._done[0])

    @done.setter
    def done(self, value):
        d = np.broadcast_to(np.asarray(value, bool), (self.num_envs,)).copy()
        self.native.set_state_host(done=d.astype(np.uint8))
        self._done = d

    @property
    def total_violations(self):
        """Lifetime violation count (base.py:57,183). Single env: host counter; batched: device counters."""
        if not self.batched:
            return self._total_violations_base
        counters, _ = self.native.read_stats()
        return int(counters[N.ST_VIOLATIONS]) + self._total_violations_base

    @total_violations.setter
    def total_violations(self, value):
        if not self.batched:
            self._total_violations_base = int(value)
            return
        counters, _ = self.native.read_stats()
        self._total_violations_base = int(value) - int(counters[N.ST_VIOLATIONS])

    def get_state(self) -> Dict[str, Any]:
        """Checkpoint: everything needed to resume bit-exactly (SoA state, counters, RNG position)."""
        s, st, vi, dn = self.native.get_state_host()
        return {"state": s, "ep_step": st, "ep_viol": vi, "done": dn, "tick": self.native.tick,
                "epoch": self.native.epoch, "seed": self.native.seed, "total_violations": self.total_violations}

    def set_state(self, ckpt: Dict[str, Any]) -> None:
        self.native.set_state_host(ckpt["state"], ckpt["ep_step"], ckpt["ep_viol"], np.asarray(ckpt["done"], np.uint8))
        self.native.set_seed(ckpt["seed"])
        self.native.set_tick(ckpt["tick"], ckpt["epoch"])
        self._state = np.array(ckpt["state"], np.float32).reshape(self.num_envs, self.state_dim)
        self._ep_step = np.asarray(ckpt["ep_step"], np.int64).copy()
        self._ep_viol = np.asarray(ckpt["ep_viol"], np.int64).copy()
        self._done = np.asarray(ckpt["done"], bool).copy()
        self.total_violations = int(ckpt.get("total_violations", 0))

    # ------------------------------------------------------------------ info
    def _get_safety_info(self, state: np.ndarray) -> Dict[str, Any]:
        """base.py:126-131"""
        return {"safety_metrics": {}, "constraint_values": {}}

    def _critical_bits(self) -> int:
        bits = 0
        for k, c in enumerate(self.safety_constraints):
            if c.critical:
                bits |= 1 << k
        return bits

    # ------------------------------------------------------------------ gym API
    def reset(self, *, seed: Optional[int] = None, options: Optional[Dict] = None) -> Tuple[np.ndarray, Dict]:
        """base.py:133-155. ``seed`` re-keys the device RNG (the reference ignores it; superset behaviour).
        ``options``: ``{"init_states": [n,S]}`` teacher-forces the initial state, ``{"mask": [n]}`` resets a subset."""
        if seed is not None:
            self.np_random = np.random.default_rng(seed)
            self.action_space.seed(seed)
            self.native.set_seed(seed)
        options = options or {}
        mask = options.get("mask")
        obs = self.native.reset_host(mask=mask, init_states=options.get("init_states"))
        if self.batched:
            self._state = obs
            info = {"total_violations": self.total_violations}
            return (obs.copy() if self.copy else obs), info
        self._state = obs.copy()
        self._ep_step[:] = 0; self._ep_viol[:] = 0; self._done[:] = False
        info = self._get_safety_info(self._state[0])
        info.update({"step": 0, "violations": 0, "total_violations": self.total_violations})
        return self._state[0].copy(), info

    def step(self, action, *, noise=None, reset_states=None):
        """base.py:157-213. ``noise`` / ``reset_states`` teacher-force the process noise (reference draw
        order) and the post-done state; omitted, both come from the in-kernel Philox streams."""
        if self._state is None:
            raise RuntimeError("Call reset() before step().")
        if self.batched:
            return self._step_batched(action, noise, reset_states)
        if self._done[0]:
            raise RuntimeError("Environment is done. Call reset() first.")       # base.py:159-160
        a = np.asarray(action, dtype=np.float32).reshape(1, self.action_dim)
        obs, next_obs, reward, flags, viol = self.native.step_host(
            a, noise=noise, reset_states=reset_states, hostmask=self._hostmask(a), want_next_obs=self.auto_reset)
        f = int(flags[0])
        terminated, truncated, critical = bool(f & N.F_TERMINATED), bool(f & N.F_TRUNCATED), bool(f & N.F_CRITICAL)
        total = len(self.safety_constraints)
        nviol = bin(int(viol[0])).count("1")
        ncrit = bin(int(viol[0]) & self._critical_bits()).count("1")
        self._ep_step[0] += 1                                                    # base.py:187
        self._ep_viol[0] += nviol                                                # base.py:182
        self._total_violations_base += nviol                                     # base.py:183
        step_out, viol_out = int(self._ep_step[0]), int(self._ep_viol[0])
        done = terminated or truncated
        self._state = obs.copy()
        final = next_obs[0].copy() if next_obs is not None else self._state[0].copy()
        if done and self.auto_reset:
            self._ep_step[0] = 0; self._ep_viol[0] = 0
        elif done:
            self._done[0] = True
        info = self._get_safety_info(final)                                      # base.py:204-211
        info.update({
            "step": step_out, "violations": viol_out, "total_violations": self.total_violations,
            "safety_metrics": SafetyMetrics(total - nviol, total, nviol, ncrit, (total - nviol) / total if total else 1.0),
            "critical_shutdown": critical,
        })
        r = np.float32(reward[0]) if self.REWARD_IS_FLOAT32 else float(reward[0])
        if self.auto_reset and done:
            info["final_observation"] = final
            return self._state[0].copy(), r, terminated, truncated, info
        return final, r, terminated, truncated, info

    def _step_batched(self, action, noise, reset_states):
        nat = self.native
        a_buf = nat.pinned("actions", (self.num_envs, self.action_dim), np.float32)
        if action is not a_buf:
            action = np.asarray(action, dtype=np.float32).reshape(self.num_envs, self.action_dim)
        hostmask = None
        if self._host_constraints():
            self._state = nat.get_state_host()[0]
            hostmask = self._hostmask(np.asarray(action))
        obs, next_obs, reward, flags, viol = nat.step_host(
            action, noise=noise, reset_states=reset_states, hostmask=hostmask, want_next_obs=self.auto_reset)
        self._state = obs
        terminated = (flags & N.F_TERMINATED) != 0
        truncated = (flags & N.F_TRUNCATED) != 0
        info = {
            "flags": flags, "violation_mask": viol, "critical_shutdown": (flags & N.F_CRITICAL) != 0,
            "safety_metrics": BatchedSafetyMetrics(viol, len(self.safety_constraints), self._critical_bits()),
        }
        if next_obs is not None:
            info["final_observation"] = next_obs
        if self.copy:
            info = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in info.items()}
            info["safety_metrics"] = BatchedSafetyMetrics(info["violation_mask"], len(self.safety_constraints), self._critical_bits())
            return obs.copy(), reward.copy(), terminated, truncated, info
        return obs, reward, terminated, truncated, info

    def rollout(self, n_steps: int, policy="random", *, steps_per_launch: int = 64, reset: bool = False, init_states=None,
                actions=None, noise=None, params=None) -> Dict[str, Any]:
        """The reference's timing / evaluation loop -- ``for _ in range(n_steps): env.step(policy(obs))`` with reset on done
        (performance_benchmark.py:106-133, utils.py:82-125) -- for every env of this object in one call: ``n_steps``
        fused in ``steps_per_launch``-step kernel launches, host arrays in and out.

        ``policy``: "random" (= ``action_space.sample()`` per step, drawn in-kernel), "zero", "dataset" with ``params``
        (the get_dataset controllers), a ``benchmarks.baseline_agents`` controller object (PID / MPC / constant / random,
        evaluated in-kernel), an ``MLPPolicy`` (a learned actor, evaluated in-kernel on the tensor cores), or "actions" with ``actions`` [T, num_envs, A] (and optionally ``noise``
        [T, num_envs, NZ]) teacher-forcing every step. Returns per-env ``reward_sum`` / ``violations`` / ``episodes``,
        the final ``obs`` and the lifetime ``stats`` (the evaluate_with_safety aggregates)."""
        nat = self.native
        if self._host_constraints():
            raise NotImplementedError("callable safety constraints cannot run inside the fused rollout kernel; "
                                      "use BoundConstraint / built-in constraints, or step()")
        pid, params = resolve_policy(nat, policy, params, actions)
        if pid == N.POLICY_ACTIONS:
            a = np.asarray(actions, np.float32).reshape(int(n_steps), self.num_envs, self.action_dim)
            actions = np.ascontiguousarray(a.transpose(0, 2, 1))            # [T, A, n]: what the kernel streams
            if noise is not None:
                z = np.asarray(noise, np.float32).reshape(int(n_steps), self.num_envs, nat.NZ)
                noise = np.ascontiguousarray(z.transpose(0, 2, 1))
        out = nat.rollout_host(n_steps, pid, steps_per_launch=steps_per_launch, params=params, init_states=init_states,
                               reset_first=reset or self._state is None, actions=actions, noise=noise)
        self._state = out["obs"]
        if not self.batched:
            self._pull()
        res = {"reward_sum": out["reward_sum"], "violations": out["violations"], "episodes": out["episodes"],
               "obs": out["obs"], "stats": nat.stats_dict(out["counters"], out["sums"])}
        if self.copy:
            res = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in res.items()}
        return res

    def get_dataset(self, quality: str = "mixed") -> Dict[str, np.ndarray]:
        raise NotImplementedError

    def render(self):
        return None

    def close(self):
        self.native.close()

    @property
    def unwrapped(self):
        return self
