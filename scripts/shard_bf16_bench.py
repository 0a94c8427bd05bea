"""Row-sharded mixed loss at BASELINE config 5 (B = 8192, T = 20, 64x64x1, K = 81 920): fp32 videos against bf16
videos, alternated in one process.

    python -m torch.distributed.run --nproc-per-node N scripts/shard_bf16_bench.py [--reps 5] [--rounds 3] [--B 8192]

Prints the card name and power limit, ms per forward + backward (device events, max over ranks), the cost_fwd stage
time, the peak memory per rank with only one dtype's inputs resident, and whether loss, terms and gradients of the
bf16 run are bit-identical to the run on the widened fp32 videos.
"""
import argparse
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kccotgan_b200.sharded import ShardedMixedLoss  # noqa: E402

HM = ("h_fake", "m_real", "h_real", "m_fake")


def card(local):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(local)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=8192)
    ap.add_argument("--T", type=int, default=20)
    ap.add_argument("--HW", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rank = dist.get_rank() if world > 1 else 0
    B, T, K = a.B, a.T, a.T * a.HW * a.HW
    sm = ShardedMixedLoss(B, K, T, 8, 1.0 / 15.0, device=dev)

    def inputs(dtype):
        g = torch.Generator(device=dev).manual_seed(1)                  # same on every rank: replicated inputs
        v = [torch.rand((B, K), generator=g, device=dev).to(torch.bfloat16).to(dtype) for _ in range(2)]
        return v + [torch.sigmoid(torch.randn((B, T, 8), generator=g, device=dev)) for _ in HM]

    def evaluate(t):
        loss, terms = sm.forward(*t)
        return loss.clone(), terms.clone(), sm.backward(1.0)

    def mx(v):
        x = torch.tensor([float(v)], device=dev)
        if world > 1:
            dist.all_reduce(x, op=dist.ReduceOp.MAX)
        return float(x)

    # peak memory: one dtype's inputs resident at a time
    peak = {}
    for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        t = inputs(dt)
        evaluate(t)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        r = evaluate(t)
        torch.cuda.synchronize()
        peak[name] = mx(torch.cuda.max_memory_allocated() / 2**30)
        del r, t
    torch.cuda.empty_cache()

    t = {"fp32": inputs(torch.float32), "bf16": inputs(torch.bfloat16)}
    out = {n: evaluate(t[n]) for n in t}                               # warm-up, and the results to compare
    torch.cuda.synchronize()
    (l16, t16, g16), (l32, t32, g32) = out["bf16"], out["fp32"]
    same = torch.equal(l16, l32) and torch.equal(t16, t32) and torch.equal(g16["fake"], g32["fake"].to(torch.bfloat16))
    same = same and all(torch.equal(g16[k], g32[k]) for k in HM)
    same = mx(0.0 if same else 1.0) == 0.0
    del out, g16, g32

    ms = {"fp32": [], "bf16": []}
    cost = {"fp32": [], "bf16": []}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(a.rounds):
        for n in ("fp32", "bf16"):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(a.reps):
                sm.forward(*t[n])
                sm.backward(1.0)
            e1.record()
            torch.cuda.synchronize()
            ms[n].append(mx(e0.elapsed_time(e1) / a.reps))
            # cost_fwd stage alone (this backend call only, no collective)
            flat = [x.reshape(B, -1) for x in t[n][:2]] + t[n][2:]
            e0.record()
            for _ in range(a.reps):
                sm.be.cost_fwd(*flat)
            e1.record()
            torch.cuda.synchronize()
            cost[n].append(mx(e0.elapsed_time(e1) / a.reps))
    if rank == 0:
        print(f"card: {card(local)}; world {world}; B={B} T={T} {a.HW}x{a.HW}x1 K={K}", flush=True)
        for n in ("fp32", "bf16"):
            print(f"{n}: fwd+bwd ms per round {[round(v, 3) for v in ms[n]]} (min {min(ms[n]):.3f}); cost_fwd ms "
                  f"{[round(v, 3) for v in cost[n]]} (min {min(cost[n]):.3f}); peak {peak[n]:.3f} GiB per rank", flush=True)
        print(f"bf16 bit-identical to widened fp32 on every rank: {same}", flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
