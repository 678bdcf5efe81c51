"""Throughput of NIG_POLICY_MLP (a learned 2-hidden-layer actor inside the fused rollout, on the tensor cores) against the
same network as a bf16 torch module driving TorchIndustrialEnv.capture_graph (one env launch per step plus the module's
own launches), alternated in one process. CUDA events around each timed pass; a 256 MiB write between timed passes
flushes the 126 MB L2 (outside the event brackets), as bench.py does.

MMA FLOP/s are computed from the shapes: padded = what the kernel issues (M = 128-row tiles, K padded to 16, the output
to N = 16), unpadded = 2 * (S*H + H*H + H*A) per env-step; both as a share of the 2,250 TFLOP/s dense-BF16 data-sheet
figure of one B200 (a data-sheet number, not a measured peak).

    python tools/mlp_rollout_bench.py [--out profiles/r03_a_mlp_rollout_bench.txt]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "neorl-industrial-gym_b200")]

import numpy as np  # noqa: E402

PEAK_BF16 = 2.25e15
K = 64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def actor(torch, S, A, H, seed=0):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Linear(S, H), torch.nn.ReLU(), torch.nn.Linear(H, H), torch.nn.ReLU(),
                               torch.nn.Linear(H, A), torch.nn.Tanh())


def flops(S, A, H):
    sp = (S + 15) // 16 * 16
    return 2 * (sp * H + H * H + H * 16), 2 * (S * H + H * H + H * A)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--steps", type=int, default=256, help="env-steps per env per timed pass (K = 64 per launch)")
    args = ap.parse_args()
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ids = {0: "ChemicalReactor-v0", 1: "PowerGrid-v0"}
    lines = [f"card: {card()}", f"K = {K}, {args.steps} env-steps per env per timed pass, best of {args.passes} passes, "
             f"L2 flushed between passes"]
    rows = []
    for kind, n in ((0, 65_536), (0, 1_048_576), (1, 1_048_576)):
        for H in (64, 256):
            env = ni.NativeEnv(kind, n, device=0, seed=1)
            env.reset_host()
            net = actor(torch, env.S, env.A, H).to(dev)
            mlp = ni.MLPPolicy.from_torch(net)
            env.set_mlp_policy(mlp)
            tenv = ni.TorchIndustrialEnv(ids[kind], n, seed=1)
            tenv.reset()
            net16 = actor(torch, env.S, env.A, H).to(dev).to(torch.bfloat16)
            with torch.no_grad():
                replay = tenv.capture_graph(lambda o: net16(o.to(torch.bfloat16)).float(), K)
                best = {"mlp": float("inf"), "torch": float("inf")}
                for p in range(args.passes + 1):           # pass 0 warms up (module load, graph capture, upload)
                    for arm in ("mlp", "torch"):
                        flush.fill_(p & 0xFF)
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        if arm == "mlp":
                            env.rollout_steps_device(args.steps, K, N.POLICY_MLP)
                        else:
                            for _ in range(args.steps // K):
                                replay()
                        e1.record()
                        torch.cuda.synchronize()
                        if p > 0:
                            best[arm] = min(best[arm], e0.elapsed_time(e1) / 1e3)
            pad, unpad = flops(env.S, env.A, H)
            steps = n * args.steps
            r = {"env": ids[kind], "n": n, "H": H, "mlp_env_steps_per_s": steps / best["mlp"],
                 "torch_graph_env_steps_per_s": steps / best["torch"], "speedup": best["torch"] / best["mlp"],
                 "mma_tflops_padded": pad * steps / best["mlp"] / 1e12, "mma_tflops_unpadded": unpad * steps / best["mlp"] / 1e12}
            r["share_of_bf16_peak_padded"] = r["mma_tflops_padded"] * 1e12 / PEAK_BF16
            r["share_of_bf16_peak_unpadded"] = r["mma_tflops_unpadded"] * 1e12 / PEAK_BF16
            rows.append(r)
            lines.append(f"{ids[kind]:20s} n={n:>9,} H={H:3d}: MLP rollout {r['mlp_env_steps_per_s']:.3e} env-steps/s, "
                         f"torch graph {r['torch_graph_env_steps_per_s']:.3e} ({r['speedup']:.1f}x); MMA "
                         f"{r['mma_tflops_padded']:.1f} TFLOP/s padded ({100 * r['share_of_bf16_peak_padded']:.2f} %), "
                         f"{r['mma_tflops_unpadded']:.1f} unpadded ({100 * r['share_of_bf16_peak_unpadded']:.2f} %)")
            print(lines[-1], flush=True)
            env.close(); tenv.close()
            del replay
            torch.cuda.empty_cache()
    text = "\n".join(lines) + "\n" + json.dumps(rows) + "\n"
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)
    print(text)


if __name__ == "__main__":
    main()
