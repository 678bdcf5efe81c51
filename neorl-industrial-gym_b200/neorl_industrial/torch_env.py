"""``TorchIndustrialEnv``: the batched env with torch CUDA tensors in and out -- no host copies at all.

For training loops whose policy already lives on the GPU: ``reset()`` / ``step(actions)`` follow the gym
signature of the reference (environments/base.py:133-213) with a leading env axis, every array is a torch tensor on
the env's device (``obs [n, S]`` fp32, ``reward [n]`` fp32, ``terminated`` / ``truncated [n]`` bool), and each call is
exactly one kernel launch on torch's current stream. Auto-reset is on: a finished env is re-initialised inside the
same launch; ``info["final_observation"]`` holds s' of the finished transition. ``capture_graph()`` records K steps
driven by a policy callable into a CUDA graph (device-resident tick) and returns a replay function; ``rollout()`` runs K steps
of an in-kernel policy (or teacher-forced actions) as one fused launch and returns every step's tuple as [K, n, ...] tensors.
"""
from __future__ import annotations

from typing import Any, Callable, Dict, Optional, Tuple

from . import _native as N
from .rollouts import resolve_policy
from .vector import KIND_BY_ID, NativeEnv


class TorchIndustrialEnv:
    def __init__(self, env_id: str, num_envs: int, *, device="cuda", seed: int = 0, env_id_offset: int = 0,
                 max_episode_steps: Optional[int] = None, constraints=None, final_observation: bool = True):
        import torch
        if env_id not in KIND_BY_ID:
            raise ValueError(f"Unknown environment '{env_id}'. Available: {', '.join(KIND_BY_ID)}")
        self.native = NativeEnv(KIND_BY_ID[env_id], num_envs, device=device, seed=seed, auto_reset=True,
                                max_episode_steps=max_episode_steps, env_id_offset=env_id_offset, constraints=constraints)
        nat = self.native
        self.env_id, self.num_envs = env_id, int(num_envs)
        self.state_dim, self.action_dim = nat.S, nat.A
        self.device = nat.torch_device()
        n = self.num_envs
        # caller-visible result buffers (AoS, exact size): overwritten by every step
        self._obs = torch.empty((n, nat.S), dtype=torch.float32, device=self.device)
        self._final = torch.empty((n, nat.S), dtype=torch.float32, device=self.device) if final_observation else None
        self._reward = torch.empty((nat.pitch,), dtype=torch.float32, device=self.device)
        self._flags = torch.empty((nat.pitch,), dtype=torch.uint8, device=self.device)
        self._viol = torch.empty((nat.pitch,), dtype=torch.uint8, device=self.device)
        self._term = torch.zeros((nat.pitch,), dtype=torch.bool, device=self.device)     # written as 0/1 bytes by the kernel
        self._trunc = torch.zeros((nat.pitch,), dtype=torch.bool, device=self.device)

    # ------------------------------------------------------------------ gym-style API on device tensors
    def reset(self, *, seed: Optional[int] = None, mask=None):
        """-> (obs [n, S], info). ``mask`` ([n] uint8/bool tensor) resets a subset."""
        import torch
        nat = self.native
        if seed is not None:
            nat.set_seed(seed)
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        nat.reset_device(mask=mask)
        nat.get_state_device(self._obs, layout=N.LAYOUT_AOS)
        return self._obs, {}

    def step(self, actions) -> Tuple[Any, Any, Any, Any, Dict[str, Any]]:
        """``actions`` [n, A] fp32 CUDA tensor (clipped to [-1, 1] in-kernel) -> obs, reward, terminated, truncated, info."""
        nat = self.native
        if not actions.dtype.is_floating_point or tuple(actions.shape) != (self.num_envs, self.action_dim):
            raise ValueError(f"actions must be a float tensor of shape ({self.num_envs}, {self.action_dim})")
        a = actions if (actions.dtype == self._obs.dtype and actions.device == self.device and actions.is_contiguous()) \
            else actions.to(device=self.device, dtype=self._obs.dtype).contiguous()
        nat.step_device(a, obs=self._obs, next_obs=self._final, reward=self._reward, flags=self._flags,
                        viol_mask=self._viol, action_layout=N.LAYOUT_AOS, aux_layout=N.LAYOUT_AOS,
                        terminated=self._term, truncated=self._trunc)
        n = self.num_envs
        # one kernel launch, no follow-up torch ops: every result is a view of a buffer the kernel wrote
        # (info["flags"] carries NIG_F_CRITICAL = 4 for the critical-shutdown bit, base.py:210)
        info = {"flags": self._flags[:n], "violation_mask": self._viol[:n]}
        if self._final is not None:
            info["final_observation"] = self._final
        return self._obs, self._reward[:n], self._term[:n], self._trunc[:n], info

    # rollout()'s keys -> nig_trajectory_t fields (the names of step()'s return and info)
    ROLLOUT_KEYS = {"obs": "obs", "actions": "actions", "rewards": "rewards", "terminated": "terminated",
                    "truncated": "truncated", "final_observation": "next_obs", "flags": "flags", "violation_mask": "viol_mask"}

    def rollout(self, n_steps: int, policy="random", *, params=None, actions=None, out=None) -> Dict[str, Any]:
        """``n_steps`` iterations of ``obs -> policy(obs) -> step`` recorded step by step in ONE fused kernel launch
        (nig_rollout_record), continuing from the current state. Returns time-major CUDA tensors: obs [T, n, S] (the
        observation the policy acted on), actions [T, n, A] (before the env's clip), rewards [T, n], terminated / truncated
        [T, n] bool, final_observation [T, n, S] (s' before the auto-reset), flags / violation_mask [T, n] uint8 -- what a loop
        of ``step`` calls that stores every result holds. The observation buffer of ``step`` / ``reset`` then holds the current
        state, so a following ``step`` carries on seamlessly. ``policy`` as in ``IndustrialEnv.rollout`` and evaluated inside
        the kernel: "random", "zero", "dataset" with ``params``, a baseline agent, an ``MLPPolicy``; or ``actions`` [T, n, A]
        teacher-forces every step. ``out`` (optional): preallocated tensors under any of these keys, filled in place."""
        import torch
        nat, n, T = self.native, self.num_envs, int(n_steps)
        pid, params = resolve_policy(nat, policy, params, actions)
        a_dev = None
        if pid == N.POLICY_ACTIONS:
            if not torch.is_tensor(actions) or tuple(actions.shape) != (T, n, self.action_dim):
                raise ValueError(f"actions must be a tensor of shape ({T}, {n}, {self.action_dim})")
            a_dev = torch.zeros((T, self.action_dim, nat.pitch), dtype=torch.float32, device=self.device)
            a_dev[:, :, :n] = actions.to(device=self.device, dtype=torch.float32).transpose(1, 2)   # [T][A][pitch]: the kernel's rows
        out = dict(out or {})
        for key in out:
            if key not in self.ROLLOUT_KEYS:
                raise ValueError(f"unknown rollout output {key!r}; expected a subset of {sorted(self.ROLLOUT_KEYS)}")
        shapes = {"obs": (T, n, self.state_dim), "actions": (T, n, self.action_dim), "final_observation": (T, n, self.state_dim)}
        dtypes = {"terminated": torch.bool, "truncated": torch.bool, "flags": torch.uint8, "violation_mask": torch.uint8}
        for key in self.ROLLOUT_KEYS:
            if out.get(key) is None:
                out[key] = torch.empty(shapes.get(key, (T, n)), dtype=dtypes.get(key, torch.float32), device=self.device)
        nat.rollout_record_device(T, pid, out={f: out[k] for k, f in self.ROLLOUT_KEYS.items()}, actions=a_dev, params=params)
        nat.get_state_device(self._obs, layout=N.LAYOUT_AOS)
        return out

    def capture_graph(self, policy: Callable, n_steps: int):
        """Record ``n_steps`` iterations of ``obs -> policy(obs) -> step`` into a CUDA graph (the policy must be
        graph-capturable torch code). Returns ``replay()``; every replay advances the env by ``n_steps`` with fresh
        process noise (device-resident tick, nig_use_device_tick). Results of the last step stay in the env's buffers."""
        import torch
        self.native.use_device_tick(2)                      # base + sequence offsets: see nig_use_device_tick
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):                       # warm-up outside capture
            out = self.step(policy(self._obs))
        torch.cuda.current_stream(self.device).wait_stream(side)
        self.native.commit_ticks()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(n_steps):
                out = self.step(policy(self._obs))
            self.native.commit_ticks()                      # last node: the base moves on by n_steps per replay
        self._graph_out = out

        def replay():
            g.replay()
            return self._graph_out
        return replay

    def stats(self) -> Dict[str, Any]:
        return self.native.stats_dict()

    def close(self):
        self.native.close()
