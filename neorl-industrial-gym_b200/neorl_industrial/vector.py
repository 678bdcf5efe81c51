"""``NativeEnv``: one libnig_b200 handle = N envs of one kind resident on one B200.

Thin, explicit wrapper over the C ABI (include/nig_b200.h). Two families of calls:
  * ``*_host``  -- numpy in / numpy out through page-locked buffers (what the gym-style API uses);
  * device      -- torch CUDA tensors by pointer on torch's current stream (zero copies; what the
                   rollout / dataset / bench paths use). torch is imported lazily and only here.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _native as N

KIND_BY_ID = {"ChemicalReactor-v0": N.ENV_CHEMICAL_REACTOR, "PowerGrid-v0": N.ENV_POWER_GRID,
              "RobotAssembly-v0": N.ENV_ROBOT_ASSEMBLY}


def _device_index(device) -> int:
    if device is None:
        return 0
    if isinstance(device, int):
        return device
    s = str(device)
    if s in ("cuda", "gpu"):
        return 0
    if s.startswith("cuda:"):
        return int(s.split(":", 1)[1])
    raise ValueError(f"device must be a CUDA device ('cuda', 'cuda:N' or an int); got {device!r}. "
                     "The B200 env path has no CPU implementation.")


def make_constraint(kind: int, cid: int = 0, si: int = 0, ai: int = -1, coef: float = 0.0, lo: float = 0.0,
                    hi: float = 0.0, penalty: float = 0.0, critical: bool = False) -> N.Constraint:
    return N.Constraint(kind, cid, si, ai, coef, lo, hi, penalty, int(bool(critical)))


class _CudaView:
    """Exposes library-owned device memory through __cuda_array_interface__ (for torch.as_tensor)."""

    def __init__(self, ptr: int, shape, typestr: str, owner):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}
        self._owner = owner


class NativeEnv:
    def __init__(self, kind: int, num_envs: int, *, device=0, seed: int = 0, auto_reset: bool = True,
                 max_episode_steps: Optional[int] = None, env_id_offset: int = 0, constraints=None):
        self._h = None
        lib = N.lib()
        self.kind = int(kind)
        spec = N.env_spec(self.kind)
        self.S, self.A, self.NZ = spec.state_dim, spec.action_dim, spec.noise_dim
        self.default_max_episode_steps = spec.max_episode_steps
        self.builtin = [spec.constraints[k] for k in range(spec.n_constraints)]
        self.n = int(num_envs)
        self.device = _device_index(device)
        cfg = N.Config()
        cfg.env_kind = self.kind
        cfg.device = self.device
        cfg.n_envs = self.n
        cfg.env_id_offset = int(env_id_offset)
        cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        cfg.max_episode_steps = 0 if max_episode_steps is None else int(max_episode_steps)
        cfg.auto_reset = int(bool(auto_reset))
        if constraints is None:
            cfg.n_constraints = -1
        else:
            if len(constraints) > N.MAX_CONSTRAINTS:
                raise ValueError(f"at most {N.MAX_CONSTRAINTS} constraints are supported")
            cfg.n_constraints = len(constraints)
            for k, c in enumerate(constraints):
                cfg.constraints[k] = c
        h = C.c_void_p()
        N.check(lib.nig_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.pitch = int(lib.nig_pitch(h))
        self.max_episode_steps = cfg.max_episode_steps or self.default_max_episode_steps
        self.auto_reset = bool(auto_reset)
        self.seed = int(seed)
        self.env_id_offset = int(env_id_offset)
        self.n_constraints = 3 if constraints is None else len(constraints)
        self._pinned = {}
        self._pinned_by_name = {}

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None):
            N.lib().nig_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def pinned(self, name: str, shape, dtype) -> np.ndarray:
        """Page-locked host array owned by this env, one per (name, shape, dtype); the lookup by name alone is the fast
        path of the single-env gym API (a few microseconds matter there)."""
        hit = self._pinned_by_name.get(name)
        if hit is not None and hit[1] == shape and hit[2] is dtype:
            return hit[0]
        key = (name, tuple(int(x) for x in np.atleast_1d(shape)), np.dtype(dtype).str)
        if key not in self._pinned:
            self._pinned[key] = N.PinnedArray(shape, dtype)
        arr = self._pinned[key].array
        self._pinned_by_name[name] = (arr, shape, dtype)
        return arr

    def set_constraints(self, constraints):
        arr = (N.Constraint * max(len(constraints), 1))(*constraints)
        N.check(N.lib().nig_set_constraints(self._h, arr, len(constraints)))
        self.n_constraints = len(constraints)

    def set_seed(self, seed: int):
        N.check(N.lib().nig_set_seed(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF))
        self.seed = int(seed)

    @property
    def tick(self) -> int:
        t, e = C.c_uint32(), C.c_uint32()
        N.check(N.lib().nig_get_tick(self._h, C.byref(t), C.byref(e)))
        return t.value

    @property
    def epoch(self) -> int:
        t, e = C.c_uint32(), C.c_uint32()
        N.check(N.lib().nig_get_tick(self._h, C.byref(t), C.byref(e)))
        return e.value

    def set_tick(self, tick: int, epoch: Optional[int] = None):
        N.check(N.lib().nig_set_tick(self._h, int(tick), self.epoch if epoch is None else int(epoch)))

    def use_device_tick(self, enable=True):
        """Device-resident step counter for CUDA-graph capture (nig_use_device_tick): ``True`` / 1 = advanced by every launch;
        2 = base + per-launch sequence offsets (lowest launch latency; end the captured sequence with ``commit_ticks()``);
        ``False`` / 0 = back to the host counter."""
        N.check(N.lib().nig_use_device_tick(self._h, int(enable)))

    def commit_ticks(self, stream=None):
        """Mode-2 device tick: move the base on by the launches made since the last commit (capture this as the last node)."""
        N.check(N.lib().nig_commit_ticks(self._h, self._stream(stream)))

    def reset_policy_state(self, stream=None):
        """Zero the device-resident PID controller state (= constructing a new PIDControllerAgent)."""
        N.check(N.lib().nig_reset_policy_state(self._h, self._stream(stream)))

    def set_mlp_policy(self, mlp):
        """Upload an ``MLPPolicy`` for NIG_POLICY_MLP (nig_set_mlp_policy: synchronises the device, invalidates captured graphs)."""
        N.check(N.lib().nig_set_mlp_policy(self._h, C.byref(mlp.native_struct())))
        self._mlp = mlp

    def use_mlp_policy(self, mlp):
        """``set_mlp_policy`` unless this very network object is already uploaded (one upload per network object)."""
        if getattr(self, "_mlp", None) is not mlp:
            self.set_mlp_policy(mlp)

    def selftest_mlp(self, obs) -> np.ndarray:
        """The uploaded network evaluated by the rollout's device code on host observations [n, S] -> actions [n, A]."""
        obs = np.ascontiguousarray(obs, np.float32).reshape(-1, self.S)
        out = np.empty((obs.shape[0], self.A), np.float32)
        N.check(N.lib().nig_selftest_mlp(self._h, obs.ctypes.data, obs.shape[0], out.ctypes.data))
        return out

    def sync(self):
        N.check(N.lib().nig_sync(self._h))

    @property
    def launch_count(self) -> int:
        return int(N.lib().nig_launch_count(self._h))

    # ------------------------------------------------------------------ host (numpy) API
    def reset_host(self, mask=None, init_states=None, want_obs=True):
        if mask is not None:
            mask = np.ascontiguousarray(mask, np.uint8).reshape(self.n)
        if init_states is not None:
            init_states = np.ascontiguousarray(init_states, np.float32).reshape(self.n, self.S)
        obs = self.pinned("obs", (self.n, self.S), np.float32) if want_obs else None
        N.check(N.lib().nig_reset_host(self._h, N.ptr_of(mask), N.ptr_of(init_states), N.ptr_of(obs)))
        return obs

    def step_host(self, actions, *, noise=None, reset_states=None, hostmask=None, want_next_obs=False, want_obs=True):
        """One step with host arrays: actions [n, A] -> (obs [n,S], next_obs|None, reward [n], flags [n], viol_mask [n]).
        The returned arrays are views of page-locked buffers that the next call overwrites."""
        a_in = self.pinned("actions", (self.n, self.A), np.float32)
        if actions is not a_in:
            np.copyto(a_in, np.asarray(actions, dtype=np.float32).reshape(self.n, self.A), casting="same_kind")
        io = N.StepIO()
        io.actions = N.ptr_of(a_in)
        if noise is not None:
            nz = self.pinned("noise", (self.n, max(self.NZ, 1)), np.float32)
            np.copyto(nz, np.asarray(noise, np.float32).reshape(self.n, self.NZ))
            io.noise = N.ptr_of(nz)
        if reset_states is not None:
            rs = self.pinned("reset_states", (self.n, self.S), np.float32)
            np.copyto(rs, np.asarray(reset_states, np.float32).reshape(self.n, self.S))
            io.reset_states = N.ptr_of(rs)
        if hostmask is not None:
            hm = self.pinned("hostmask", (self.n,), np.uint8)
            np.copyto(hm, np.asarray(hostmask, np.uint8).reshape(self.n))
            io.hostmask = N.ptr_of(hm)
        obs = self.pinned("obs", (self.n, self.S), np.float32) if want_obs else None
        next_obs = self.pinned("next_obs", (self.n, self.S), np.float32) if want_next_obs else None
        reward = self.pinned("reward", (self.n,), np.float32)
        flags = self.pinned("flags", (self.n,), np.uint8)
        viol = self.pinned("viol", (self.n,), np.uint8)
        io.obs, io.next_obs = N.ptr_of(obs), N.ptr_of(next_obs)
        io.reward, io.flags, io.viol_mask = N.ptr_of(reward), N.ptr_of(flags), N.ptr_of(viol)
        io.action_layout = io.aux_layout = N.LAYOUT_AOS
        N.check(N.lib().nig_step_host(self._h, C.byref(io)))
        return obs, next_obs, reward, flags, viol

    def rollout_host(self, n_steps: int, policy: int = N.POLICY_UNIFORM, *, steps_per_launch: int = 64, params=None,
                     init_states=None, reset_first: bool = False, actions=None, noise=None, want_obs: bool = True):
        """``n_steps`` env-steps per env in ceil(n_steps / steps_per_launch) fused launches with HOST buffers in and out
        (nig_rollout_host). ``actions`` [T, A, n] / ``noise`` [T, NZ, n] teacher-force the run (policy ACTIONS).
        Returns a dict of page-locked arrays (overwritten by the next call): reward_sum [n], violations [n],
        episodes [n], obs [n, S], counters [24], sums [8]."""
        r = N.RolloutHost()
        r.n_steps, r.steps_per_launch, r.policy, r.reset_first = int(n_steps), int(steps_per_launch), int(policy), int(bool(reset_first))
        keep = []
        if init_states is not None:
            buf = self.pinned("init_states", (self.n, self.S), np.float32)
            if init_states is not buf:
                np.copyto(buf, np.asarray(init_states, np.float32).reshape(self.n, self.S))
            r.init_states = N.ptr_of(buf)
        if actions is not None:
            a = np.ascontiguousarray(actions, np.float32).reshape(int(n_steps), self.A, self.n)
            keep.append(a)
            r.actions = N.ptr_of(a)
        if noise is not None:
            z = np.ascontiguousarray(noise, np.float32).reshape(int(n_steps), self.NZ, self.n)
            keep.append(z)
            r.noise = N.ptr_of(z)
        if params is not None:
            r.pp = params
        out = {"reward_sum": self.pinned("ro_reward", (self.n,), np.float32),
               "violations": self.pinned("ro_viol", (self.n,), np.int32),
               "episodes": self.pinned("ro_done", (self.n,), np.int32),
               "counters": self.pinned("ro_counters", (24,), np.int64),
               "sums": self.pinned("ro_sums", (8,), np.float64)}
        r.reward_sum, r.viol_count, r.done_count = N.ptr_of(out["reward_sum"]), N.ptr_of(out["violations"]), N.ptr_of(out["episodes"])
        r.counters24, r.sums8 = N.ptr_of(out["counters"]), N.ptr_of(out["sums"])
        if want_obs:
            out["obs"] = self.pinned("obs", (self.n, self.S), np.float32)
            r.final_obs = N.ptr_of(out["obs"])
        N.check(N.lib().nig_rollout_host(self._h, C.byref(r)))
        return out

    def get_state_host(self):
        state = np.empty((self.n, self.S), np.float32)
        step = np.empty(self.n, np.int32)
        viol = np.empty(self.n, np.int32)
        done = np.empty(self.n, np.uint8)
        N.check(N.lib().nig_get_state_host(self._h, N.ptr_of(state), N.ptr_of(step), N.ptr_of(viol), N.ptr_of(done)))
        return state, step, viol, done.astype(bool)

    def set_state_host(self, state=None, ep_step=None, ep_viol=None, done=None):
        if state is not None:
            state = np.ascontiguousarray(state, np.float32).reshape(self.n, self.S)
        if ep_step is not None:
            ep_step = np.ascontiguousarray(ep_step, np.int32).reshape(self.n)
        if ep_viol is not None:
            ep_viol = np.ascontiguousarray(ep_viol, np.int32).reshape(self.n)
        if done is not None:
            done = np.ascontiguousarray(done, np.uint8).reshape(self.n)
        N.check(N.lib().nig_set_state_host(self._h, N.ptr_of(state), N.ptr_of(ep_step), N.ptr_of(ep_viol), N.ptr_of(done)))

    def read_stats(self):
        counters = np.zeros(24, np.int64)
        sums = np.zeros(8, np.float64)
        N.check(N.lib().nig_read_stats(self._h, N.ptr_of(counters), N.ptr_of(sums)))
        return counters, sums

    def track_returns(self, on: bool = True):
        """Whether the single-step kernels keep the per-env episode-return accumulator (on by default: finished-episode
        return statistics stay correct when ``step`` and ``rollout`` calls are mixed). Off saves 16 B of HBM traffic per
        env-step; the statistics then cover only episodes that ran entirely inside rollout calls."""
        N.check(N.lib().nig_track_returns(self._h, int(bool(on))))

    def track_step_stats(self, on: bool = True):
        """Whether single steps add to the device counter block (``stats_dict``); off saves ~1 us per launch at 65,536 envs.
        The per-env outputs of ``step`` and the fused rollouts' counters are not affected."""
        N.check(N.lib().nig_track_step_stats(self._h, int(bool(on))))

    def track_extrema(self, on: bool = True):
        """Rollouts of this handle also keep the smallest / largest finished-episode return (a 2 % slower kernel flavour)."""
        N.check(N.lib().nig_track_extrema(self._h, int(bool(on))))

    def read_extrema(self):
        """(return_min, return_max) over the episodes finished inside rollouts since the last clear_stats, or (None, None)."""
        lo, hi, have = C.c_double(), C.c_double(), C.c_int32()
        N.check(N.lib().nig_read_extrema(self._h, C.byref(lo), C.byref(hi), C.byref(have)))
        return (lo.value, hi.value) if have.value else (None, None)

    def extrema_tensor(self):
        """Zero-copy torch view int64[2] of the extremum keys (combine across ranks with all_reduce(MAX), then decode_extrema)."""
        import torch
        p = C.c_void_p()
        N.check(N.lib().nig_extrema_ptr(self._h, C.byref(p)))
        return torch.as_tensor(_CudaView(p.value, (2,), "<i8", self), device=self.torch_device())

    @staticmethod
    def decode_extrema(keys):
        k = np.ascontiguousarray(keys, np.int64)
        lo, hi, have = C.c_double(), C.c_double(), C.c_int32()
        N.check(N.lib().nig_decode_extrema(N.ptr_of(k), C.byref(lo), C.byref(hi), C.byref(have)))
        return (lo.value, hi.value) if have.value else (None, None)

    def stats_dict(self, counters=None, sums=None):
        if counters is None:
            counters, sums = self.read_stats()
        d = {"steps": int(counters[N.ST_STEPS]), "episodes": int(counters[N.ST_EPISODES]),
             "terminated": int(counters[N.ST_TERMINATED]), "truncated": int(counters[N.ST_TRUNCATED]),
             "critical_shutdowns": int(counters[N.ST_CRITICAL]), "violations": int(counters[N.ST_VIOLATIONS]),
             "successes": int(counters[N.ST_SUCCESSES]), "episode_length_sum": int(counters[N.ST_EP_LEN_SUM]),
             "episode_length_sq": int(counters[N.ST_EP_LEN_SQ]),
             "violations_per_constraint": [int(counters[N.ST_CON0 + k]) for k in range(self.n_constraints)],
             "return_sum": float(sums[0]), "return_sq": float(sums[1]), "reward_sum": float(sums[2])}
        return d

    def clear_stats(self, stream=None):
        N.check(N.lib().nig_clear_stats(self._h, self._stream(stream)))

    # ------------------------------------------------------------------ device (torch) API
    @staticmethod
    def _stream(stream=None):
        if stream is not None:
            return int(stream)
        import torch
        return int(torch.cuda.current_stream().cuda_stream)

    def torch_device(self):
        import torch
        return torch.device("cuda", self.device)

    def state_tensor(self):
        """Zero-copy torch view [S, pitch] fp32 of the SoA device state."""
        import torch
        sp, wp = C.c_void_p(), C.c_void_p()
        N.check(N.lib().nig_state_ptr(self._h, C.byref(sp), C.byref(wp)))
        return torch.as_tensor(_CudaView(sp.value, (self.S, self.pitch), "<f4", self), device=self.torch_device())

    def stats_tensor(self):
        """Zero-copy torch view of the device stats block as int64[32] (slots >= 24 hold fp64 bit patterns); the shard copies
        the plain single-step kernel adds to are folded in on the current stream first (nig_fold_stats)."""
        import torch
        p = C.c_void_p()
        N.check(N.lib().nig_fold_stats(self._h, self._stream()))
        N.check(N.lib().nig_stats_ptr(self._h, C.byref(p)))
        return torch.as_tensor(_CudaView(p.value, (N.STATS_SLOTS,), "<i8", self), device=self.torch_device())

    def empty(self, rows: Optional[int] = None, dtype=None):
        """Device buffer sized for per-env arrays: [pitch] or [rows, pitch]."""
        import torch
        dtype = dtype or torch.float32
        shape = (self.pitch,) if rows is None else (rows, self.pitch)
        return torch.zeros(shape, dtype=dtype, device=self.torch_device())

    def reset_device(self, mask=None, init_states=None, layout=N.LAYOUT_SOA, stream=None):
        N.check(N.lib().nig_reset(self._h, N.ptr_of(mask), N.ptr_of(init_states), layout, self._stream(stream)))

    def step_device(self, actions, *, noise=None, reset_states=None, hostmask=None, obs=None, next_obs=None,
                    reward=None, flags=None, viol_mask=None, action_layout=N.LAYOUT_SOA, aux_layout=N.LAYOUT_SOA,
                    terminated=None, truncated=None, stream=None):
        io = N.StepIO()
        io.actions, io.noise, io.reset_states = N.ptr_of(actions), N.ptr_of(noise), N.ptr_of(reset_states)
        io.hostmask = N.ptr_of(hostmask)
        io.obs, io.next_obs, io.reward = N.ptr_of(obs), N.ptr_of(next_obs), N.ptr_of(reward)
        io.flags, io.viol_mask = N.ptr_of(flags), N.ptr_of(viol_mask)
        io.action_layout, io.aux_layout = action_layout, aux_layout
        io.terminated, io.truncated = N.ptr_of(terminated), N.ptr_of(truncated)
        N.check(N.lib().nig_step(self._h, C.byref(io), self._stream(stream)))

    def rollout_device(self, n_steps: int, policy: int = N.POLICY_UNIFORM, *, actions=None, noise=None, params=None,
                       use_tma: bool = True, reward_sum=None, viol_count=None, done_count=None, stream=None):
        r = N.Rollout()
        r.n_steps, r.policy = int(n_steps), int(policy)
        r.flags = N.ROLLOUT_USE_TMA if (use_tma and policy == N.POLICY_ACTIONS) else 0
        r.actions, r.noise = N.ptr_of(actions), N.ptr_of(noise)
        if params is not None:
            r.pp = params
        r.reward_sum, r.viol_count, r.done_count = N.ptr_of(reward_sum), N.ptr_of(viol_count), N.ptr_of(done_count)
        N.check(N.lib().nig_rollout(self._h, C.byref(r), self._stream(stream)))

    # nig_trajectory_t fields: (per-step width or None for [T, n] rows, accepted torch dtype names)
    RECORD_FIELDS = {"obs": ("S", ("float32",)), "actions": ("A", ("float32",)), "rewards": (None, ("float32",)),
                     "flags": (None, ("uint8",)), "viol_mask": (None, ("uint8",)), "terminated": (None, ("uint8", "bool")),
                     "truncated": (None, ("uint8", "bool")), "next_obs": ("S", ("float32",))}

    def rollout_record_device(self, n_steps: int, policy: int = N.POLICY_UNIFORM, *, out: dict, actions=None, noise=None,
                              params=None, reward_sum=None, viol_count=None, done_count=None, stream=None):
        """``rollout_device`` that also records every step (nig_rollout_record, one launch): ``out`` maps any subset of
        obs / actions / next_obs ([T, n, S | A] fp32), rewards ([T, n] fp32), flags / viol_mask ([T, n] uint8) and
        terminated / truncated ([T, n] uint8 or bool) to contiguous CUDA tensors on this env's device; row [t, i] is what
        ``step_device`` writes for env i at step t. ``actions`` [T, A, pitch] / ``noise`` [T, NZ, pitch] teacher-force the run
        (policy ACTIONS) as in ``rollout_device``. Every tensor is checked before anything is launched (ValueError)."""
        import torch
        T, dev = int(n_steps), self.torch_device()
        tr = N.Trajectory()
        for name, x in out.items():
            if name not in self.RECORD_FIELDS:
                raise ValueError(f"unknown trajectory field {name!r}; expected a subset of {sorted(self.RECORD_FIELDS)}")
            if x is None:
                continue
            width, dtypes = self.RECORD_FIELDS[name]
            shape = (T, self.n) if width is None else (T, self.n, getattr(self, width))
            if not isinstance(x, torch.Tensor) or x.device != dev:
                raise ValueError(f"out[{name!r}] must be a torch tensor on {dev}")
            if str(x.dtype).replace("torch.", "") not in dtypes:
                raise ValueError(f"out[{name!r}] must have dtype {' or '.join(dtypes)}, not {x.dtype}")
            if tuple(x.shape) != shape:
                raise ValueError(f"out[{name!r}] must have shape {shape}, not {tuple(x.shape)}")
            if not x.is_contiguous():
                raise ValueError(f"out[{name!r}] must be contiguous")
            setattr(tr, name, x.data_ptr())
        r = N.Rollout()
        r.n_steps, r.policy = T, int(policy)
        r.actions, r.noise = N.ptr_of(actions), N.ptr_of(noise)
        if params is not None:
            r.pp = params
        r.reward_sum, r.viol_count, r.done_count = N.ptr_of(reward_sum), N.ptr_of(viol_count), N.ptr_of(done_count)
        N.check(N.lib().nig_rollout_record(self._h, C.byref(r), C.byref(tr), self._stream(stream)))

    def rollout_steps_device(self, total_steps: int, steps_per_launch: int = 64, policy: int = N.POLICY_UNIFORM, *, params=None,
                             reward_sum=None, viol_count=None, done_count=None, accumulate: bool = False, stream=None):
        """``total_steps`` steps of every env in ``steps_per_launch``-step fused launches with an in-kernel policy; large
        populations advance as env slices on internal streams (nig_rollout_steps). Asynchronous on ``stream``."""
        r = N.Rollout()
        r.n_steps, r.policy = int(steps_per_launch), int(policy)
        r.flags = N.ROLLOUT_ACCUMULATE if accumulate else 0
        if params is not None:
            r.pp = params
        r.reward_sum, r.viol_count, r.done_count = N.ptr_of(reward_sum), N.ptr_of(viol_count), N.ptr_of(done_count)
        N.check(N.lib().nig_rollout_steps(self._h, C.byref(r), int(total_steps), self._stream(stream)))

    def get_state_device(self, state=None, layout=N.LAYOUT_SOA, ep_step=None, ep_viol=None, done=None, stream=None):
        N.check(N.lib().nig_get_state(self._h, N.ptr_of(state), layout, N.ptr_of(ep_step), N.ptr_of(ep_viol),
                                      N.ptr_of(done), self._stream(stream)))

    def set_state_device(self, state=None, layout=N.LAYOUT_SOA, ep_step=None, ep_viol=None, done=None, stream=None):
        N.check(N.lib().nig_set_state(self._h, N.ptr_of(state), layout, N.ptr_of(ep_step), N.ptr_of(ep_viol),
                                      N.ptr_of(done), self._stream(stream)))

    def dataset_device(self, n_episodes: int, n_steps: int, policy: int, params, out: dict, capacity: int,
                       terminals_include_truncation: bool = True, stream=None) -> int:
        d = N.DatasetOut()
        d.observations, d.actions, d.rewards = N.ptr_of(out["observations"]), N.ptr_of(out["actions"]), N.ptr_of(out["rewards"])
        d.terminals, d.timeouts = N.ptr_of(out["terminals"]), N.ptr_of(out.get("timeouts"))
        d.next_observations, d.safety = N.ptr_of(out.get("next_observations")), N.ptr_of(out.get("safety"))
        d.capacity = int(capacity)
        d.terminals_include_truncation = int(bool(terminals_include_truncation))
        nw = C.c_int64(0)
        N.check(N.lib().nig_dataset(self._h, int(n_episodes), int(n_steps), int(policy), C.byref(params), C.byref(d),
                                    C.byref(nw), self._stream(stream)))
        return nw.value

    def dataset_size(self, n_episodes: int, n_steps: int, policy: int, params, stream=None) -> int:
        nt = C.c_int64(0)
        N.check(N.lib().nig_dataset_size(self._h, int(n_episodes), int(n_steps), int(policy), C.byref(params),
                                         C.byref(nt), self._stream(stream)))
        return nt.value
