"""torchrun worker of tests/test_sharded_nccl_ctx.py: the row-sharded mixed loss with shared context frames
(ctx_frames > 0) over N GPUs against the fp64 oracle of the WHOLE problem.  Inputs are uniform with the first ctx frames
of `fake` copied from `real`; the gathered `fake` gradient is compared on the predicted frames and must be exactly zero
on the context frames.

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29631 \
        tests/sharded_nccl_ctx_worker.py [B T H W C ctx]
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
    B, T, H, W, C, ctx = (a + [1024, 4, 16, 16, 1, 2][len(a):])[:6]
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rank = dist.get_rank() if world > 1 else 0
    s = 1.0 / 15.0
    inp = make_inputs(B=B, T=T, H=H, W=W, C=C, J=8, kind="uniform", seed=1)      # same on every rank
    inp["fake"][:, :, :ctx] = inp["real"][:, :, :ctx]
    t = [inp[k].to(dev) for k in NAMES]
    sm = ShardedMixedLoss(B, T * H * W * C, T, 8, s, device=dev, ctx_frames=ctx)
    loss, terms = sm.forward(*t)
    g = sm.backward(1.0)
    torch.cuda.synchronize()
    full = {}
    for k in ("fake", "h_fake", "h_real"):
        if world > 1:
            parts = [torch.empty_like(g[k]) for _ in range(world)]
            dist.all_gather(parts, g[k].contiguous())
            full[k] = torch.cat(parts, 0)
        else:
            full[k] = g[k]
    if rank == 0:
        from oracle import closed_form as cf
        npin = [inp[k].double().numpy() for k in NAMES]
        ref, gref, det = cf.compute_sinkhorn_loss(npin[0], npin[1], s, 0.8, 100, *npin[2:], video=True, grad=True)
        ref_terms = np.array([det["loss_xy"], det["loss_xx"], det["loss_yy"]])
        scale = np.abs(ref_terms).max()
        terr = np.abs(terms.double().cpu().numpy() - ref_terms).max() / scale
        lerr = abs(float(loss) - ref) / scale
        gf = full["fake"].double().cpu().numpy()
        errs = {"fake": float(np.linalg.norm(gf[:, :, ctx:] - gref["f_fake"][:, :, ctx:]) /
                              np.linalg.norm(gref["f_fake"][:, :, ctx:]))}
        for k in ("h_fake", "h_real", "m_real", "m_fake"):
            got = (full[k] if k in full else g[k]).double().cpu().numpy().reshape(gref[k].shape)
            errs[k] = float(np.linalg.norm(got - gref[k]) / np.linalg.norm(gref[k]))
        zero = bool((gf[:, :, :ctx] == 0).all())
        ok = terr <= 1e-4 and lerr <= 1e-4 and all(e <= 1e-4 for e in errs.values()) and zero
        print(f"world={world} B={B} K={T * H * W * C} ctx={ctx}: terms err {terr:.2e} loss err {lerr:.2e} grads {errs} "
              f"context gradient zero: {zero}", flush=True)
        print("SHARDED_CTX_OK" if ok else "SHARDED_CTX_FAIL", flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
