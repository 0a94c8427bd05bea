"""torchrun worker of tests/test_sharded_nccl_bf16.py: the row-sharded mixed loss on bf16 videos over N GPUs.

On every rank the bf16 evaluation must equal the evaluation on the widened fp32 videos (loss, terms and h / m
gradients bit for bit, the `fake` rows the fp32 rows rounded to nearest even); rank 0 checks the gathered result
against the fp64 oracle of the whole problem on the bf16-rounded inputs.

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29621 \
        tests/sharded_nccl_bf16_worker.py [B T H W C]
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kccotgan_b200.sharded import ShardedMixedLoss  # noqa: E402
from kccotgan_b200.synthetic import make_inputs  # noqa: E402

NAMES = ("real", "fake", "h_fake", "m_real", "h_real", "m_fake")


def main():
    a = [int(v) for v in sys.argv[1:]]
    B, T, H, W, C = (a + [1024, 4, 16, 16, 1][len(a):])[:5]
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rank = dist.get_rank() if world > 1 else 0
    s = 1.0 / 15.0
    inp = make_inputs(B=B, T=T, H=H, W=W, C=C, J=8, kind="uniform", seed=1)      # same on every rank
    inp["real"], inp["fake"] = inp["real"].bfloat16(), inp["fake"].bfloat16()
    t16 = [inp[k].to(dev) for k in NAMES]
    t32 = [t.float() for t in t16]
    sm = ShardedMixedLoss(B, T * H * W * C, T, 8, s, device=dev)
    res = {}
    for name, t in (("bf16", t16), ("fp32", t32)):
        loss, terms = sm.forward(*t)
        res[name] = (loss.clone(), terms.clone(), sm.backward(1.0))
    torch.cuda.synchronize()
    (l16, t16_, g16), (l32, t32_, g32) = res["bf16"], res["fp32"]
    ok = torch.equal(l16, l32) and torch.equal(t16_, t32_) and g16["fake"].dtype == torch.bfloat16
    ok = ok and torch.equal(g16["fake"], g32["fake"].to(torch.bfloat16))
    ok = ok and all(torch.equal(g16[k], g32[k]) for k in ("h_fake", "m_real", "h_real", "m_fake"))
    flag = torch.tensor([0 if ok else 1], device=dev)
    if world > 1:
        dist.all_reduce(flag)
    print(f"rank {rank}: bf16 == widened fp32: {ok}", flush=True)
    full = {}
    for k in ("fake", "h_fake", "h_real"):
        if world > 1:
            parts = [torch.empty_like(g16[k]) for _ in range(world)]
            dist.all_gather(parts, g16[k].contiguous())
            full[k] = torch.cat(parts, 0)
        else:
            full[k] = g16[k]
    if rank == 0:
        from oracle import closed_form as cf
        npin = [inp[k].double().numpy() for k in NAMES]
        ref, gref, det = cf.compute_sinkhorn_loss(npin[0], npin[1], s, 0.8, 100, *npin[2:], video=True, grad=True)
        ref_terms = np.array([det["loss_xy"], det["loss_xx"], det["loss_yy"]])
        scale = np.abs(ref_terms).max()
        terr = np.abs(t16_.double().cpu().numpy() - ref_terms).max() / scale
        lerr = abs(float(l16) - ref) / scale
        errs = {}
        for k, n in (("fake", "f_fake"), ("h_fake", "h_fake"), ("h_real", "h_real"), ("m_real", "m_real"),
                     ("m_fake", "m_fake")):
            got = (full[k] if k in full else g16[k]).double().cpu().numpy().reshape(gref[n].shape)
            errs[k] = float(np.linalg.norm(got - gref[n]) / np.linalg.norm(gref[n]))
        oracle_ok = terr <= 1e-4 and lerr <= 1e-4 and errs["fake"] <= 4e-3 and \
            all(e <= 1e-4 for k, e in errs.items() if k != "fake")
        print(f"world={world} B={B} K={T * H * W * C}: terms err {terr:.2e} loss err {lerr:.2e} grads {errs}", flush=True)
        print("SHARDED_BF16_OK" if oracle_ok and int(flag) == 0 else "SHARDED_BF16_FAIL", flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
