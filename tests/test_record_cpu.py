"""nig_rollout_record without a GPU: the ctypes mirror of nig_trajectory_t against include/nig_b200.h compiled by the host
compiler, the ABI version, the bound symbol, and the policy parsing that IndustrialEnv.rollout and TorchIndustrialEnv.rollout
share."""
import ctypes as C
import os
import subprocess

import pytest

from neorl_industrial import _native as N
from neorl_industrial.rollouts import resolve_policy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_trajectory_struct_matches_header(tmp_path):
    fields = [f for f, _ in N.Trajectory._fields_]
    src = tmp_path / "traj.c"
    offs = ", ".join(f"offsetof(nig_trajectory_t, {f})" for f in fields)
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "nig_b200.h"\n'
                   'int main(void){size_t o[] = {' + offs + '}; printf("%zu %d", sizeof(nig_trajectory_t), NIG_ABI_VERSION);'
                   ' for (size_t k = 0; k < sizeof o / sizeof o[0]; ++k) printf(" %zu", o[k]); printf("\\n"); return 0;}\n')
    exe = tmp_path / "traj"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    want = [C.sizeof(N.Trajectory), N.ABI_VERSION] + [getattr(N.Trajectory, f).offset for f in fields]
    assert got == want, (got, want)
    assert fields == ["obs", "actions", "rewards", "flags", "viol_mask", "terminated", "truncated", "next_obs"]
    assert N.ABI_VERSION == 6
    res, args = N.SYMBOLS["nig_rollout_record"]
    assert res is C.c_int and args[1] == C.POINTER(N.Rollout) and args[2] == C.POINTER(N.Trajectory)


class _Nat:
    def __init__(self):
        self.uploaded = []

    def use_mlp_policy(self, m):
        self.uploaded.append(m)


def test_resolve_policy():
    import numpy as np
    import neorl_industrial as ni
    from neorl_industrial.benchmarks import BaselineAgentFactory
    nat = _Nat()
    assert resolve_policy(nat, "random") == (N.POLICY_UNIFORM, None)
    assert resolve_policy(nat, "uniform") == (N.POLICY_UNIFORM, None)
    assert resolve_policy(nat, "zero") == (N.POLICY_ZERO, None)
    pp = N.PolicyParams()
    assert resolve_policy(nat, "dataset", pp) == (N.POLICY_PCTRL, pp)
    assert resolve_policy(nat, "random", None, actions=np.zeros((2, 3, 1))) == (N.POLICY_ACTIONS, None)
    pid, bp = resolve_policy(nat, BaselineAgentFactory.create("mpc", 12, 3))
    assert pid == N.POLICY_BASELINE and bp.baseline.kind == N.BASELINE_MPC
    mlp = ni.MLPPolicy([np.zeros((64, 12), np.float32), np.zeros((3, 64), np.float32)])
    assert resolve_policy(nat, mlp) == (N.POLICY_MLP, None) and nat.uploaded == [mlp]
    with pytest.raises(ValueError, match="needs an actions array"):
        resolve_policy(nat, "actions")
    with pytest.raises(ValueError, match="needs PolicyParams"):
        resolve_policy(nat, "dataset")
    with pytest.raises(ValueError, match="unknown rollout policy"):
        resolve_policy(nat, "greedy")
