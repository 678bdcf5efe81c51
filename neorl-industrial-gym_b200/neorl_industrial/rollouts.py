"""Batched evaluation loops: the ``reset -> while not done: step`` loops of utils.evaluate_with_safety
(utils.py:82-154) and OfflineAgent.evaluate (agents/base.py:330-393) over N envs at once.

Two flavours:
  * ``evaluate_policy_device``: the policy runs inside the fused rollout kernel (uniform random, zero, the
    get_dataset P-controllers, a learned ``MLPPolicy``) -- no host round trips; aggregates come from the device stats block, which
    ``distributed.allreduce_stats`` can sum across GPUs.
  * ``evaluate_agent_batched``: an arbitrary ``agent.predict(obs, deterministic=True)`` callback drives the
    batched ``env.step`` (host arrays).
Both return the reference's result keys.
"""
from __future__ import annotations

import math
from typing import Any, Dict, Optional

import numpy as np

from . import _native as N
from .policies import MLPPolicy


ROLLOUT_POLICY_IDS = {"random": N.POLICY_UNIFORM, "uniform": N.POLICY_UNIFORM, "zero": N.POLICY_ZERO}


def resolve_policy(nat, policy, params=None, actions=None):
    """The ``policy`` argument of ``IndustrialEnv.rollout`` and ``TorchIndustrialEnv.rollout`` -> (NIG_POLICY_* id, params):
    "random" / "uniform" / "zero", "dataset" with ``params`` (the get_dataset controllers), a ``benchmarks.baseline_agents``
    controller object, an ``MLPPolicy`` (uploaded to ``nat`` once per network object), or teacher-forced ``actions``
    (``policy="actions"`` or any policy with ``actions`` given; the caller lays them out for the kernel)."""
    if actions is not None or policy == "actions":
        if actions is None:
            raise ValueError("policy='actions' needs an actions array [T, num_envs, A]")
        return N.POLICY_ACTIONS, params
    if hasattr(policy, "device_policy"):                   # benchmarks.baseline_agents controllers, in-kernel
        return policy.device_policy()
    if isinstance(policy, MLPPolicy):                      # a learned actor on the tensor cores, in-kernel
        nat.use_mlp_policy(policy)
        return N.POLICY_MLP, params
    if policy == "dataset":
        if params is None:
            raise ValueError("policy='dataset' needs PolicyParams (see datasets.policy_params)")
        return N.POLICY_PCTRL, params
    try:
        return ROLLOUT_POLICY_IDS[policy], params
    except KeyError:
        raise ValueError(f"unknown rollout policy {policy!r}; expected one of "
                         f"{sorted(ROLLOUT_POLICY_IDS) + ['dataset', 'actions']}") from None


def metrics_from_stats(stats: Dict[str, Any], n_constraints: int, critical_flags) -> Dict[str, Any]:
    """Reference result dict (utils.py:128-152) from summed device counters."""
    ep = max(int(stats["episodes"]), 1)
    steps = max(int(stats["steps"]), 1)
    mean = stats["return_sum"] / ep
    var = max(stats["return_sq"] / ep - mean * mean, 0.0)
    lmean = stats["episode_length_sum"] / ep
    lvar = max(stats["episode_length_sq"] / ep - lmean * lmean, 0.0)
    per_con = stats["violations_per_constraint"]
    crit = sum(int(v) for v, c in zip(per_con, critical_flags) if c)
    return {
        "return_mean": mean, "return_std": math.sqrt(var), "return_min": None, "return_max": None,
        "length_mean": lmean, "length_std": math.sqrt(lvar),
        "safety_violations": int(stats["violations"]), "safety_violations_per_episode": stats["violations"] / ep,
        "critical_violations": crit, "emergency_shutdowns": int(stats["critical_shutdowns"]),
        "constraint_satisfaction_rate": 1.0 - stats["violations"] / (steps * max(n_constraints, 1)),
        "successful_episodes": int(stats["successes"]), "success_rate": stats["successes"] / ep,
        "episodes": int(stats["episodes"]), "steps": int(stats["steps"]),
    }


def evaluate_policy_device(env, n_steps: int, policy: int = N.POLICY_UNIFORM, params=None, *, chunk: int = 64,
                           reduce_fn=None) -> Dict[str, Any]:
    """Run ``n_steps`` env-steps per env with an in-kernel policy (auto-reset on) and return the reference's
    evaluation keys over every episode that finished. ``reduce_fn(counters, sums) -> (counters, sums)`` hooks in the
    cross-GPU all-reduce (see distributed.allreduce_stats). ``policy`` may also be an ``MLPPolicy``: the learned actor runs
    inside the kernel (NIG_POLICY_MLP), uploaded once per network object."""
    nat = env.native
    if isinstance(policy, MLPPolicy):
        nat.use_mlp_policy(policy)
        policy = N.POLICY_MLP
    nat.clear_stats()
    nat.track_extrema(True)            # the kernel flavour that also keeps return_min / return_max
    try:
        nat.rollout_steps_device(n_steps, chunk, policy, params=params)    # chunk-step fused launches, env slices on streams
    finally:
        nat.track_extrema(False)
    counters, sums = nat.read_stats()
    if reduce_fn is not None:
        counters, sums = reduce_fn(counters, sums)
    stats = nat.stats_dict(counters, sums)
    out = metrics_from_stats(stats, len(env.safety_constraints), [c.critical for c in env.safety_constraints])
    # return_min / return_max of this rank's episodes; across ranks: distributed.allreduce_extrema(nat)
    out["return_min"], out["return_max"] = nat.read_extrema()
    return out


def evaluate_agent_batched(agent: Any, env: Any, n_episodes: int = 100) -> Dict[str, Any]:
    """utils.py:82-154 with a batched env. The reference runs ``n_episodes`` episodes one after the other, each from a fresh
    reset to its end; here the episodes are dealt out to the envs as QUOTAS -- env i runs its first
    ``n_episodes // num_envs`` (+1 for the first ``n_episodes % num_envs`` envs) episodes to the end and only those count,
    every step of them and nothing else. (Keeping "the first n_episodes to finish across all envs" instead would favour
    short episodes: the sample would be biased towards early terminations.)"""
    if not getattr(env, "auto_reset", False):
        raise ValueError("batched evaluation needs an auto-resetting env (ni.make(..., num_envs=N))")
    n = env.num_envs
    quota = np.full(n, n_episodes // n, np.int64)
    quota[: n_episodes % n] += 1
    finished = np.zeros(n, np.int64)
    obs, _ = env.reset()
    ep_ret = np.zeros(n, np.float64)
    ep_len = np.zeros(n, np.int64)
    returns, lengths = [], []
    viol = crit = shut = 0
    sat_sum, sat_n = 0.0, 0
    while np.any(finished < quota):
        live = finished < quota                      # envs still inside their quota: only their steps are counted
        action = np.asarray(agent.predict(obs, deterministic=True), np.float32).reshape(n, env.action_dim)
        obs, reward, terminated, truncated, info = env.step(action)
        ep_ret += reward
        ep_len += 1
        sm = info["safety_metrics"]
        viol += int(np.asarray(sm.violation_count)[live].sum()); crit += int(np.asarray(sm.critical_violations)[live].sum())
        sat_sum += float(np.asarray(sm.satisfaction_rate, np.float64)[live].sum()); sat_n += int(live.sum())
        shut += int(np.sum(np.asarray(info["critical_shutdown"])[live]))
        done = (terminated | truncated)
        for i in np.flatnonzero(done & live):
            returns.append(float(ep_ret[i])); lengths.append(int(ep_len[i]))
        finished[done & live] += 1
        ep_ret[done] = 0.0; ep_len[done] = 0
    returns, lengths = np.array(returns), np.array(lengths)
    succ = int(np.sum(returns > 0))
    return {
        "return_mean": returns.mean(), "return_std": returns.std(), "return_min": returns.min(), "return_max": returns.max(),
        "length_mean": lengths.mean(), "length_std": lengths.std(),
        "safety_violations": viol, "safety_violations_per_episode": viol / n_episodes, "critical_violations": crit,
        "emergency_shutdowns": shut, "constraint_satisfaction_rate": (sat_sum / sat_n) if sat_n else 1.0,
        "successful_episodes": succ, "success_rate": succ / n_episodes,
    }
