"""T4/T5 on CPU: the multi-GPU host logic under torch.distributed `gloo`, world_size 2.
  * problem-parallel partitioning (no collective on the data path);
  * the fused row-sharded mixed loss (cost shift, cost partials, adjoint panels and gradient sums
    exchanged between ranks), with an fp64 CPU stand-in for the kernels, against the single-process oracle."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def test_split_problems_covers_everything():
    from kccotgan_b200.sharded import row_range, split_problems
    for nprob in (1, 7, 256, 257):
        for world in (1, 2, 3, 8):
            seen = []
            for r in range(world):
                seen += list(split_problems(nprob, r, world))
            assert seen == list(range(nprob))
            sizes = [len(split_problems(nprob, r, world)) for r in range(world)]
            assert max(sizes) - min(sizes) <= 1
    assert row_range(8192, 3, 8) == (3072, 4096)


def _mixed_worker(rank, world, port, shape, inp, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from kccotgan_b200.sharded import ShardedMixedLoss, row_range
        from _shard_cpu_backend import CpuMixedShardBackend
        B, T, D, J = shape
        r0, r1 = row_range(B, rank, world)
        be = CpuMixedShardBackend(B, T * D, T, J, 1.0 / 15.0, 1.0, 100, r0, r1 - r0)
        sm = ShardedMixedLoss(B, T * D, T, J, 1.0 / 15.0, backend=be)
        t = [torch.from_numpy(a) for a in inp]
        loss, terms = sm.forward(*t)
        g = sm.backward(1.0)
        out[rank] = (float(loss), terms.numpy(), {k: v.numpy() for k, v in g.items()}, r0, r1)
    finally:
        dist.destroy_process_group()


def test_row_sharded_mixed_loss_two_ranks():
    """The fused row-sharded loss (cost rows -> sharded Sinkhorn -> all-to-all of the adjoint panels -> gradient
    rows) on 2 gloo ranks with the fp64 CPU stand-in for the kernels, against the single-process oracle."""
    from oracle import closed_form as cf
    rng = np.random.default_rng(3)
    B, T, D, J = 12, 4, 6, 3
    real, fake = rng.random((B, T, D)), rng.random((B, T, D))
    hm = [1.0 / (1.0 + np.exp(-rng.standard_normal((B, T, J)))) for _ in range(4)]
    inp = [real, fake] + hm
    mgr = mp.Manager()
    out = mgr.dict()
    port = 29500 + ((os.getpid() + 7) % 2000)
    mp.spawn(_mixed_worker, args=(2, port, (B, T, D, J), inp, out), nprocs=2, join=True)
    ref, gref, det = cf.compute_sinkhorn_loss(real, fake, 1.0 / 15.0, 0.8, 100, *hm, video=False, grad=True)
    ref_terms = np.array([det["loss_xy"], det["loss_xx"], det["loss_yy"]])
    rows = {k: np.zeros_like(gref[n]) for k, n in (("fake", "f_fake"), ("h_fake", "h_fake"), ("h_real", "h_real"))}
    for rank in (0, 1):
        loss, terms, g, r0, r1 = out[rank]
        assert abs(loss - ref) < 1e-9 * np.abs(ref_terms).max()
        assert np.abs(terms - ref_terms).max() < 1e-9 * np.abs(ref_terms).max()
        for k in rows:
            rows[k][r0:r1] = g[k]
        for k, n in (("m_real", "m_real"), ("m_fake", "m_fake")):      # replicated after the all-reduce
            assert np.linalg.norm(g[k] - gref[n]) < 1e-8 * np.linalg.norm(gref[n]), k
    for k, n in (("fake", "f_fake"), ("h_fake", "h_fake"), ("h_real", "h_real")):
        assert np.linalg.norm(rows[k] - gref[n]) < 1e-8 * np.linalg.norm(gref[n]), k
