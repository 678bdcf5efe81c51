"""Throughput of nig_rollout_record (the fused rollout that writes every step's obs / action / reward / terminated /
truncated into [K, n, ...] device tensors) against the caller's own loop that collects the same tensors: TorchIndustrialEnv
stepping into preallocated [K, n, ...] buffers, captured as a CUDA graph (device-resident tick), with the same policy --
uniform random actions drawn by torch, or the same 2-hidden-layer network as a bf16 torch module (as tools/mlp_rollout_bench.py).
The arms alternate in one process; CUDA events around each timed pass, a 256 MiB write between passes flushes the 126 MB L2
(outside the event brackets). Bytes written by the record kernel are computed from the shapes: (4 S + 4 A + 4 + 1 + 1) per
env-step. The device-to-device copy bandwidth of a 4 GiB torch copy (read + write bytes) is measured in the same process as
the yardstick of the record kernel's write bandwidth.

    python tools/record_bench.py [--out profiles/r03_c_record_bench.txt]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "neorl-industrial-gym_b200")]

K = 64
FIELDS = ("obs", "actions", "rewards", "terminated", "truncated")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def actor(torch, S, A, H, seed=0):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Linear(S, H), torch.nn.ReLU(), torch.nn.Linear(H, H), torch.nn.ReLU(),
                               torch.nn.Linear(H, A), torch.nn.Tanh())


def buffers(torch, dev, n, S, A):
    return {"obs": torch.empty((K, n, S), device=dev), "actions": torch.empty((K, n, A), device=dev),
            "rewards": torch.empty((K, n), device=dev), "terminated": torch.empty((K, n), dtype=torch.bool, device=dev),
            "truncated": torch.empty((K, n), dtype=torch.bool, device=dev)}


def graph_loop(torch, tenv, policy, bufs):
    """K iterations of obs -> policy -> step with every result copied into the [K, n, ...] buffers, as one CUDA graph."""
    nat, cur = tenv.native, torch.cuda.current_stream()
    nat.use_device_tick(2)

    def body():
        obs = tenv._obs
        for t in range(K):
            a = policy(obs)
            bufs["obs"][t].copy_(obs)
            bufs["actions"][t].copy_(a)
            obs, r, te, tr, _ = tenv.step(a)
            bufs["rewards"][t].copy_(r)
            bufs["terminated"][t].copy_(te)
            bufs["truncated"][t].copy_(tr)
    side = torch.cuda.Stream()
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        body()                                     # warm-up outside the capture
    cur.wait_stream(side)
    nat.commit_ticks()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        body()
        nat.commit_ticks()
    return g.replay


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--launches", type=int, default=4, help="K-step launches (record) / graph replays (torch) per timed pass")
    args = ap.parse_args()
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(fn, p):
        flush.fill_(p & 0xFF)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.launches):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3

    x = torch.empty(4 << 30, dtype=torch.uint8, device=dev)
    y = torch.empty_like(x)
    copy = []
    for p in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); y.copy_(x); e1.record(); torch.cuda.synchronize()
        if p:
            copy.append(2 * x.numel() / (e0.elapsed_time(e1) / 1e3))
    copy_bw = max(copy)
    del x, y
    lines = [f"card: {card()}", f"K = {K}, {args.launches} launches / replays per timed pass, best of {args.passes} passes, "
             f"L2 flushed between passes; recorded fields {', '.join(FIELDS)}",
             f"device-to-device copy (torch, 4 GiB, read + write bytes): {copy_bw / 1e9:.0f} GB/s"]
    print("\n".join(lines), flush=True)
    ids = {0: "ChemicalReactor-v0", 1: "PowerGrid-v0"}
    rows = []
    for kind, n in ((0, 65_536), (0, 1_048_576), (1, 1_048_576)):
        for H in (None, 64, 256):
            env = ni.NativeEnv(kind, n, device=0, seed=1)
            env.reset_host()
            S, A = env.S, env.A
            tenv = ni.TorchIndustrialEnv(ids[kind], n, seed=1, final_observation=False)
            tenv.reset()
            if H is None:
                pid, policy = N.POLICY_UNIFORM, (lambda o: torch.rand((n, A), device=dev) * 2 - 1)
            else:
                env.set_mlp_policy(ni.MLPPolicy.from_torch(actor(torch, S, A, H).to(dev)))
                net16 = actor(torch, S, A, H).to(dev).to(torch.bfloat16)
                pid, policy = N.POLICY_MLP, (lambda o: net16(o.to(torch.bfloat16)).float())
            rec = buffers(torch, dev, n, S, A)
            rec = {k: (v.view(torch.uint8) if v.dtype == torch.bool else v) for k, v in rec.items()}
            col = buffers(torch, dev, n, S, A)
            with torch.no_grad():
                replay = graph_loop(torch, tenv, policy, col)
                best = {"record": float("inf"), "torch": float("inf")}
                for p in range(args.passes + 1):              # pass 0 warms up
                    for arm in ("record", "torch"):
                        fn = (lambda: env.rollout_record_device(K, pid, out=rec)) if arm == "record" else replay
                        t = timed(fn, p)
                        if p:
                            best[arm] = min(best[arm], t)
            steps = n * K * args.launches
            bpe = 4 * S + 4 * A + 4 + 1 + 1
            r = {"env": ids[kind], "n": n, "policy": "uniform" if H is None else f"mlp H={H}", "bytes_per_env_step": bpe,
                 "record_env_steps_per_s": steps / best["record"], "torch_graph_env_steps_per_s": steps / best["torch"],
                 "speedup": best["torch"] / best["record"]}
            r["record_write_gbs"] = bpe * r["record_env_steps_per_s"] / 1e9
            r["share_of_copy_bw"] = r["record_write_gbs"] * 1e9 / copy_bw
            rows.append(r)
            lines.append(f"{ids[kind]:20s} n={n:>9,} {r['policy']:10s}: record {r['record_env_steps_per_s']:.3e} env-steps/s, "
                         f"{r['record_write_gbs']:.0f} GB/s written ({100 * r['share_of_copy_bw']:.0f} % of the copy), "
                         f"torch graph loop {r['torch_graph_env_steps_per_s']:.3e} ({r['speedup']:.1f}x)")
            print(lines[-1], flush=True)
            env.close(); tenv.close()
            del replay, rec, col
            torch.cuda.empty_cache()
    text = "\n".join(lines) + "\n" + json.dumps(rows) + "\n"
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)
    print(text)


if __name__ == "__main__":
    main()
