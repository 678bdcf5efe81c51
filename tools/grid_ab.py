"""PowerGrid-v0 / RobotAssembly-v0 fused rollout throughput (uniform policy, K = 64, 256 steps per pass):
   python tools/grid_ab.py [kind=1] [n_envs ...]    (NIG_GRID_FAST = 0 generic kernel / 1 the dedicated kernel)"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "neorl-industrial-gym_b200")]
import numpy as np, torch
import neorl_industrial as ni
from neorl_industrial import _native as N

def run(kind, n, horizon=256, K=64, reps=7, sliced=False):
    env = ni.NativeEnv(kind, n, device=0, seed=0)
    env.reset_device()
    def one_pass():
        if sliced:
            env.rollout_steps_device(horizon, K, N.POLICY_UNIFORM)
        else:
            for _ in range(horizon // K): env.rollout_device(K, N.POLICY_UNIFORM)
    for _ in range(2): one_pass()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); one_pass(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    st = env.stats_dict()
    env.close()
    return n * horizon / (np.median(ts) * 1e-3), st["return_sum"], st["episodes"]

if __name__ == "__main__":
    kind = int(sys.argv[1]) if len(sys.argv) > 1 else 1
    ns = [int(x) for x in sys.argv[2:]] or [1 << 20]
    for n in ns:
        for sliced in (False, True):
            v, ret, ep = run(kind, n, sliced=sliced)
            print(f"kind={kind} NIG_GRID_FAST={os.environ.get('NIG_GRID_FAST', 'default')} n={n:8d} {'slices' if sliced else 'single'} "
                  f"{v:.4g} env-steps/s  return_sum {ret:.9e} episodes {ep}", flush=True)
