"""The single-step kernel at the BASELINE population (65,536 reactor envs): eager and graph-replayed launch time.
   env knob: NIG_STEP_VEC (1/2/4); argv: [n_envs] [track_returns 0/1] [step_counters 0/1]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "neorl-industrial-gym_b200")]
import torch
import neorl_industrial as ni
from neorl_industrial import _native as N
n = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
track = int(sys.argv[2]) if len(sys.argv) > 2 else 1
counters = int(sys.argv[3]) if len(sys.argv) > 3 else 1
dev = torch.device("cuda", 0)
env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=0, seed=0)
env.track_returns(bool(track))
env.track_step_stats(bool(counters))
env.reset_device()
acts = torch.rand((3, env.pitch), device=dev) * 2 - 1
rew, fl, vm = env.empty(), env.empty(dtype=torch.uint8), env.empty(dtype=torch.uint8)
for _ in range(50):
    env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(1000):
    env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
e1.record(); torch.cuda.synchronize()
eager = e0.elapsed_time(e1)
mode = int(os.environ.get("TICK_MODE", "2"))
env.use_device_tick(mode)
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    for _ in range(100):
        env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
    env.commit_ticks()
g.replay(); torch.cuda.synchronize()
e0.record()
for _ in range(10):
    g.replay()
e1.record(); torch.cuda.synchronize()
graph = e0.elapsed_time(e1)
print(f"tick_mode={mode} n={n} vec={os.environ.get('NIG_STEP_VEC', 'auto')} track_returns={track} step_counters={counters}: "
      f"eager {eager:.3f} us/launch, graph {graph:.3f} us/launch", flush=True)
