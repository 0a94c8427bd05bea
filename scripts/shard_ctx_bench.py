"""Row-sharded mixed loss at BASELINE config 5 (B = 8192, T = 20 with 10 context frames, 64x64x1, K = 81 920): the
plain call against the shared-context call (ctx_frames = 10), fp32 and bf16 videos, alternated in one process.

    python -m torch.distributed.run --nproc-per-node N scripts/shard_ctx_bench.py [--reps 5] [--rounds 3] [--B 8192]

Prints the card name and power limit, ms per forward + backward (device events, max over ranks), the cost_fwd and
cost_bwd stage times, the peak memory per rank of each variant on its own, the tensor-core work of the cost GEMMs of
both variants, and how far the hinted results are from the plain ones on the same inputs (fake's first 10 frames are
real's, as in kernel_train.py:268).
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


def gemm_flops(B, Brows, K, period, clen):
    """executed MMA flops of this rank's cost GEMMs (3 fp16 products, k padded to 64-column blocks):
    forward = the three Brows x B blocks, backward = the fake adjoint Brows x K over the 2B stacked rows"""
    pad = lambda v: (v + 63) // 64 * 64                                    # noqa: E731
    R = 2 * B
    f = lambda m, n, k: 3 * 2 * m * n * k                                   # noqa: E731
    plain = (3 * f(Brows, B, pad(K)), f(Brows, K, pad(R)))
    if not clen:
        return plain
    nc = K // period * clen
    nq = K - nc
    return (f(Brows, B, pad(nc)) + 3 * f(Brows, B, pad(nq)), f(Brows, nq, pad(R)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=8192)
    ap.add_argument("--T", type=int, default=20)
    ap.add_argument("--ctx", type=int, default=10)
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
    B, T, HW = a.B, a.T, a.HW
    K = T * HW * HW
    s = 1.0 / 15.0

    def make(variant):
        return ShardedMixedLoss(B, K, T, 8, s, device=dev, ctx_frames=a.ctx if variant == "ctx" else 0)

    def inputs(dtype):
        g = torch.Generator(device=dev).manual_seed(1)                  # same on every rank: replicated inputs
        real, fake = [torch.rand((B, HW, T, HW, 1), generator=g, device=dev).to(torch.bfloat16).to(dtype)
                      for _ in range(2)]
        fake[:, :, :a.ctx] = real[:, :, :a.ctx]
        return [real, fake] + [torch.sigmoid(torch.randn((B, T, 8), generator=g, device=dev)) for _ in HM]

    def evaluate(sm, t):
        loss, terms = sm.forward(*t)
        g = sm.backward(1.0)
        return loss.clone(), terms.clone(), {k: v.clone() for k, v in g.items()}

    def mx(v):
        x = torch.tensor([float(v)], device=dev)
        if world > 1:
            dist.all_reduce(x, op=dist.ReduceOp.MAX)
        return float(x)

    runs = [(v, d) for d in ("fp32", "bf16") for v in ("plain", "ctx")]
    dts = {"fp32": torch.float32, "bf16": torch.bfloat16}

    # peak memory: each variant on its own, one dtype's inputs resident
    peak = {}
    for v, d in runs:
        sm, t = make(v), inputs(dts[d])
        evaluate(sm, t)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        r = evaluate(sm, t)
        torch.cuda.synchronize()
        peak[(v, d)] = (mx(torch.cuda.max_memory_allocated() / 2**30), mx((torch.cuda.max_memory_allocated() - base) / 2**30))
        del r, t, sm
        torch.cuda.empty_cache()

    sms = {"plain": make("plain"), "ctx": make("ctx")}
    t = {d: inputs(dts[d]) for d in dts}
    out = {(v, d): evaluate(sms[v], t[d]) for v, d in runs}              # warm-up, and the results to compare
    torch.cuda.synchronize()
    diffs = {}
    for d in dts:
        (l0, t0, g0), (l1, t1, g1) = out[("plain", d)], out[("ctx", d)]
        scale = float(t0.abs().max())
        dterm = float((t1.double() - t0.double()).abs().max()) / scale
        f0, f1 = g0["fake"][:, :, a.ctx:].double(), g1["fake"][:, :, a.ctx:].double()
        dg = {"fake": float((f1 - f0).norm() / f0.norm())}
        dg.update({k: float((g1[k].double() - g0[k].double()).norm() / g0[k].double().norm()) for k in HM})
        zero = bool((g1["fake"][:, :, :a.ctx] == 0).all())
        diffs[d] = (mx(dterm), {k: mx(v) for k, v in dg.items()}, mx(0.0 if zero else 1.0) == 0.0)
    same16 = all(torch.equal(out[("ctx", "bf16")][i], out[("ctx", "fp32")][i]) for i in (0, 1))
    del out

    ms, cf, cb = ({k: [] for k in runs} for _ in range(3))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(a.reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return mx(e0.elapsed_time(e1) / a.reps)

    for _ in range(a.rounds):
        for v, d in runs:
            sm, x = sms[v], t[d]
            ms[(v, d)].append(timed(lambda: (sm.forward(*x), sm.backward(1.0))))
            # the cost stages alone (these backend calls only, no collective); cost_bwd reuses the cost adjoints of
            # the last backward and the split of the last cost_fwd, which saw the same inputs
            flat = [y.reshape(B, -1) for y in x[:2]] + x[2:]
            cf[(v, d)].append(timed(lambda: sm.be.cost_fwd(*flat)))
            XY, YY = sm._columns_of(sm.be.Cbar3[0]), sm._columns_of(sm.be.Cbar3[2])
            cb[(v, d)].append(timed(lambda: sm.be.cost_bwd(XY, YY)))
    if rank == 0:
        Brows = B // world
        fw0, bw0 = gemm_flops(B, Brows, K, T * HW, 0)
        fw1, bw1 = gemm_flops(B, Brows, K, T * HW, a.ctx * HW)
        print(f"card: {card(local)}; world {world}; B={B} T={T} ctx={a.ctx} {HW}x{HW}x1 K={K}", flush=True)
        print(f"cost GEMM MMA flops per rank: forward {fw0 / 1e12:.2f} -> {fw1 / 1e12:.2f} TFLOP ({fw1 / fw0:.3f}), "
              f"fake adjoint {bw0 / 1e12:.2f} -> {bw1 / 1e12:.2f} TFLOP ({bw1 / bw0:.3f})", flush=True)
        r = lambda xs: [round(x, 3) for x in xs]                           # noqa: E731
        for v, d in runs:
            print(f"{d} {v:5s}: fwd+bwd ms {r(ms[(v, d)])} (min {min(ms[(v, d)]):.3f}); cost_fwd ms {r(cf[(v, d)])} "
                  f"(min {min(cf[(v, d)]):.3f}); cost_bwd ms {r(cb[(v, d)])} (min {min(cb[(v, d)]):.3f}); "
                  f"peak {peak[(v, d)][0]:.3f} GiB allocated ({peak[(v, d)][1]:.3f} GiB above the resident buffers)",
                  flush=True)
        for d in dts:
            saved = min(ms[("plain", d)]) - min(ms[("ctx", d)])
            sf = min(cf[("plain", d)]) - min(cf[("ctx", d)])
            sb = min(cb[("plain", d)]) - min(cb[("ctx", d)])
            print(f"{d}: hint saves {saved:.3f} ms per fwd+bwd ({saved / min(ms[('plain', d)]):.1%}), cost_fwd "
                  f"{sf:.3f} ms ({sf / min(cf[('plain', d)]):.1%}), cost_bwd {sb:.3f} ms ({sb / min(cb[('plain', d)]):.1%})",
                  flush=True)
            dterm, dg, zero = diffs[d]
            print(f"{d}: hinted vs plain: terms {dterm:.2e} of the largest term; gradients rel-L2 "
                  + ", ".join(f"{k} {e:.2e}" for k, e in dg.items()) + f"; context gradient zero: {zero}", flush=True)
        print(f"hinted bf16 loss and terms bit-identical to hinted fp32 on the widened videos: {same16}", flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
