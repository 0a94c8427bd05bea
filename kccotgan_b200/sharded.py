"""Multi-GPU modes of the loss path (SURVEY.md §8e) — one process per GPU over torch.distributed.

1. Independent problems (BASELINE config 4, data-parallel replicas): `split_problems` deals problems
   to ranks; each rank runs the single-GPU kernels on its share; NO data-path collective.
2. One large problem (config 5): the rows of the B x B cost are sharded (`row_range`).
   `ShardedMixedLoss` computes a rank's cost rows, runs its row block of the three Sinkhorn solves in
   persistent kernels that exchange the [B] column sums with the other ranks through peer mailboxes
   (no host-launched collective per iteration), and returns the gradient rows of the rank's samples;
   NCCL carries only a few collectives per evaluation.  The backend is pluggable so that the partition /
   exchange logic is testable with `gloo` on CPU (the tests pass their own fp64 stand-in; the product
   backend is CUDA-only — there is no CPU fallback in this package).
"""
import ctypes
import math

import torch
import torch.distributed as dist

from . import _lib
from .functional import _as_dtypes, _check_hm, _videos


def split_problems(nprob, rank, world):
    """Contiguous block of problem indices for `rank` (sizes differ by at most one)."""
    base, rem = divmod(int(nprob), int(world))
    start = rank * base + min(rank, rem)
    return range(start, start + base + (1 if rank < rem else 0))


def row_range(B, rank, world):
    """Rows [r0, r1) of the cost matrix owned by `rank`."""
    r = split_problems(B, rank, world)
    return r.start, r.stop


# ------------------------------------------------------------------------------------------------
# Fused row-sharded mixed loss (BASELINE config 5 on N GPUs): cost rows, persistent Sinkhorn with the
# in-kernel mailbox exchange, gradient rows.  gan_utils.py:204-227 on one problem spread over the ranks.
# ------------------------------------------------------------------------------------------------
class PeerMailbox:
    """The peer-mapped memory the persistent Sinkhorn kernels exchange their column sums through: one mailbox
    and one flag array per rank, allocated with torch's symmetric memory (CUDA VMM handles exchanged over the
    process group) so that every rank holds device pointers to every other rank's copy."""

    def __init__(self, np_, B, dev, group):
        import torch.distributed._symmetric_memory as symm
        lib = _lib.load()
        world = dist.get_world_size(group)
        self.world = world
        nfl = int(lib.kccot_shard_mailbox_bytes(np_, world, B)) // 4
        self.mbox = symm.empty(nfl, dtype=torch.float32, device=dev)
        self.flags = symm.empty(max(world, 2) * _lib.SHARD_FLAGS_PER_RANK, dtype=torch.int64, device=dev)
        self.mbox.zero_()
        self.flags.zero_()
        torch.cuda.synchronize(dev)
        pg = group if group is not None else dist.group.WORLD
        self._hm = symm.rendezvous(self.mbox, pg)
        self._hf = symm.rendezvous(self.flags, pg)
        dist.barrier(group)                                   # every rank's zeros are in place before anyone writes
        self.mbox_ptrs = (ctypes.c_void_p * world)(*[int(p) for p in self._hm.buffer_ptrs])
        self.flag_ptrs = (ctypes.c_void_p * world)(*[int(p) for p in self._hf.buffer_ptrs])
        self.launches = 0

    def next_epoch(self):
        """A fresh epoch base per persistent launch, identical on all ranks (they launch in lock step)."""
        self.launches += 1
        return self.launches << 24


class CudaMixedShardBackend:
    """The C-ABI stages of the fused row-sharded loss on this rank's samples [row0, row0 + Brows).

    `cost_fwd` validates its inputs before any launch and raises ValueError for anything the kernels cannot read:
    videos and h / m must be CUDA tensors on this backend's device with [B, K] and [B, T, J] elements.  Two bf16
    videos go to the bf16 entry points (a view that is not 16-byte aligned is cloned) and `cost_bwd` then returns the
    `fake` gradient rows in bf16: the fp32 rows on the widened videos, rounded to nearest even.  A bf16 video next to
    an fp32 one, and bf16 h / m, are widened (exact).  Every other dtype is rejected.

    `ctx = (ctx_period, ctx_len)` is the shared-context hint of include/kccot.h, passed to the `_ctx` entry points: with
    ctx_len > 0 the columns c with c % ctx_period < ctx_len of `fake` are never read (the `real` values stand in) and
    the `fake` gradient rows are zero there; with ctx_len = 0 they run the plain computation.  (0, 0), the default,
    calls the plain entry points."""

    def __init__(self, B, K, T, J, s, eps, L, row0, Brows, dev, group, ctx=(0, 0)):
        self.B, self.K, self.T, self.J, self.s, self.eps, self.L = B, K, T, J, float(s), float(eps), int(L)
        self.row0, self.Brows, self.dev, self.group = row0, Brows, dev, group
        self.ctx = (int(ctx[0]), int(ctx[1]))
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        lib = _lib.load()
        f32 = dict(dtype=torch.float32, device=dev)
        if self.ctx != (0, 0):
            nb = lib.kccot_shard_cost_workspace_bytes_ctx(B, K, Brows, *self.ctx)
            if nb == 0:
                raise ValueError(f"bad shared-context hint (period, len) = {self.ctx} for K = {K}")
        else:
            nb = lib.kccot_shard_cost_workspace_bytes(B, K, Brows)
        self.ws_cost = torch.empty(nb, dtype=torch.uint8, device=dev)
        nb = lib.kccot_shard_sinkhorn_workspace_bytes(3, Brows, B, self.L)
        if nb == 0:
            raise ValueError(f"row-sharded Sinkhorn needs 64 < B <= 8192 and B % 4 == 0, got B={B}")
        self.ws_sk = torch.empty(nb, dtype=torch.uint8, device=dev)
        self.C3 = torch.empty((3, Brows, B), **f32)
        self.Cbar3 = torch.empty((3, Brows, B), **f32)
        self.u_hist = torch.empty((3, self.L + 1, B), **f32)
        self.v_hist = torch.empty((3, self.L + 1, B), **f32)
        self.nits = torch.empty(3, dtype=torch.int32, device=dev)
        self.shift = torch.empty(3, **f32)
        self.cost_partial = torch.empty((3, 2), **f32)
        self.mail = PeerMailbox(3, B, dev, group) if self.world > 1 else None

    def _st(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    @staticmethod
    def _p(t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else None

    def _comm(self):
        if self.mail is None:
            return None, None, 0
        return self.mail.mbox_ptrs, self.mail.flag_ptrs, self.mail.next_epoch()

    def _check(self, real, fake, hm):
        real, fake, bf16 = _videos(real, fake)
        hm = [_check_hm(t, n, 3) for t, n in zip(hm, ("h_fake", "m_real", "h_real", "m_fake"))]
        for t, n, shape in [(real, "f_real", (self.B, self.K)), (fake, "f_fake", (self.B, self.K))] + \
                [(t, n, (self.B, self.T, self.J)) for t, n in zip(hm, ("h_fake", "m_real", "h_real", "m_fake"))]:
            if tuple(t.shape) != shape:
                raise ValueError(f"{n}: expected shape {shape}, got {tuple(t.shape)}")
            if t.device != self.ws_cost.device:
                raise ValueError(f"{n}: expected a tensor on {self.ws_cost.device}, got {t.device}")
        return real, fake, bf16, hm

    def cost_fwd(self, real, fake, h_fake, m_real, h_real, m_fake):
        real, fake, self.bf16, hm = self._check(real, fake, (h_fake, m_real, h_real, m_fake))
        h_fake, m_real, h_real, m_fake = hm
        self.inputs = (real, fake, h_fake, m_real, h_real, m_fake)
        p = self._p
        args = (p(real), p(fake), self.B, self.K, self.row0, self.Brows, p(h_fake), p(m_real), p(h_real), p(m_fake),
                self.T, self.J, self.s, p(self.C3), p(self.ws_cost), self.ws_cost.numel(), self._st())
        name = "kccot_shard_cost_fwd_bf16" if self.bf16 else "kccot_shard_cost_fwd"
        with torch.cuda.device(self.dev):
            if self.ctx != (0, 0):
                _lib.call(name + "_ctx", *args, *self.ctx)
            else:
                _lib.call(name, *args)
            _lib.call("kccot_shard_local_min", p(self.C3), 3, self.Brows, self.B, p(self.shift), self._st())
        return self.shift

    def sinkhorn_fwd(self):
        p = self._p
        mb, fl, ep = self._comm()
        with torch.cuda.device(self.dev):
            _lib.call("kccot_shard_sinkhorn_fwd", p(self.C3), 3, self.Brows, self.B, self.row0, self.eps, self.L, 100, 1e-2, 0,
                      p(self.u_hist), p(self.v_hist), p(self.nits), p(self.cost_partial), p(self.shift), self.world, self.rank,
                      mb, fl, ep, p(self.ws_sk), self.ws_sk.numel(), self._st())
        return self.cost_partial

    def sinkhorn_bwd(self, gcost3):
        p = self._p
        mb, fl, ep = self._comm()
        with torch.cuda.device(self.dev):
            _lib.call("kccot_shard_sinkhorn_bwd", p(self.C3), 3, self.Brows, self.B, self.row0, self.eps, self.L, p(self.u_hist),
                      p(self.v_hist), p(self.nits), p(gcost3), p(self.Cbar3), p(self.shift), self.world, self.rank, mb, fl, ep,
                      p(self.ws_sk), self.ws_sk.numel(), self._st())
        return self.Cbar3

    def cost_bwd(self, XYcol, YYcol):
        p = self._p
        real, fake, h_fake, m_real, h_real, m_fake = self.inputs
        f32 = dict(dtype=torch.float32, device=self.dev)
        g_fake = torch.empty((self.Brows, self.K), dtype=torch.bfloat16 if self.bf16 else torch.float32, device=self.dev)
        gh_fake = torch.empty((self.Brows, self.T, self.J), **f32)
        gh_real = torch.empty((self.Brows, self.T, self.J), **f32)
        gm_real = torch.empty((self.B, self.T, self.J), **f32)
        gm_fake = torch.empty((self.B, self.T, self.J), **f32)
        args = (p(self.Cbar3), p(XYcol), p(YYcol), self.B, self.K, self.row0, self.Brows, p(h_fake), p(m_real),
                p(h_real), p(m_fake), self.T, self.J, self.s, p(g_fake), p(gh_fake), p(gm_real), p(gh_real), p(gm_fake),
                p(self.ws_cost), self.ws_cost.numel(), self._st())
        name = "kccot_shard_cost_bwd_bf16" if self.bf16 else "kccot_shard_cost_bwd"
        with torch.cuda.device(self.dev):
            if self.ctx != (0, 0):
                _lib.call(name + "_ctx", *args, *self.ctx)
            else:
                _lib.call(name, *args)
        return g_fake, gh_fake, gm_real, gh_real, gm_fake


class ShardedMixedLoss:
    """`compute_sinkhorn_loss` (gan_utils.py:204-227: eps = 1.0, L = 100) of ONE problem whose cost rows are
    spread over the ranks of `group`.  Every rank passes the full (replicated) tensors — real, fake [B, ...],
    h / m [B, T, J] — and owns the samples `row_range(B, rank, world)`.

    forward()  -> (loss, terms[3]) replicated on all ranks.
    backward() -> gradients of this rank's own samples: `fake` [Brows, ...] and `h_fake`, `h_real` [Brows, T, J];
                  `m_real`, `m_fake` [B, T, J] summed over ranks (every sample's M meets every row).  Each gradient
                  comes back in the dtype of its input.
    The CUDA backend takes fp32 or bf16 videos and h / m (see CudaMixedShardBackend).  With bf16 videos the results
    are exactly those of fp32 videos widened from them: loss, terms and the h / m gradients bit for bit, the `fake`
    rows the fp32 rows rounded to nearest even, with no fp32 copy of a video.  bf16 m gradients are rounded after
    the fp32 all-reduce, so every rank holds the same bits.
    `ctx_frames` > 0 states that the first ctx_frames frames of `fake` are those of `real` (kernel_train.py:268,
    fake = concat(real_in, fake_pred)).  forward() then takes [B, H, T, W, C] videos, never reads fake's context
    frames, and computes their share of the three cost blocks once; the result equals the plain one within
    floating-point tolerance, and the `fake` gradient is that of the predicted frames, zero on the context frames.
    Collectives of one evaluation (all small except the two [Brows, B] all-to-alls): MIN of 3 floats, SUM of 6
    floats, all-to-all of Cbar_xy / Cbar_yy, SUM of two [B, T, J]; the 2 x L x 3 column-sum exchanges of the
    Sinkhorn iterations happen inside the persistent kernels.
    """

    def __init__(self, B, K, T, J, scaling_coef, eps=1.0, L=100, group=None, device=None, backend=None, ctx_frames=0):
        if not 0 <= int(ctx_frames) < int(T):
            raise ValueError(f"ctx_frames must be in [0, T = {T}), got {ctx_frames}")
        if ctx_frames and backend is not None:
            raise ValueError("ctx_frames > 0 needs the CUDA backend (a user-supplied backend takes no shared-context hint)")
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        if B % self.world:
            raise ValueError(f"B = {B} must be a multiple of the number of ranks ({self.world})")
        self.B, self.K, self.T, self.J = int(B), int(K), int(T), int(J)
        self.s, self.eps, self.L = float(scaling_coef), float(eps), int(L)
        self.row0, r1 = row_range(B, self.rank, self.world)
        self.Brows = r1 - self.row0
        self.ctx_frames, self.device = int(ctx_frames), device
        if self.ctx_frames:
            self.be = None                  # the hint needs the videos' frame size: the backend is made by forward()
        else:
            self.be = backend if backend is not None else CudaMixedShardBackend(
                self.B, self.K, self.T, self.J, self.s, self.eps, self.L, self.row0, self.Brows, device, group)

    def _allreduce(self, t, op):
        if self.world > 1:
            dist.all_reduce(t, op=op, group=self.group)
        return t

    def _columns_of(self, rows):
        """[Brows, B] row panel on every rank -> [B, Brows] column panel: out[i, jl] = M[i, row0 + jl]."""
        if self.world == 1:
            return rows.contiguous()
        N, Br = self.world, self.Brows
        send = rows.reshape(Br, N, Br).permute(1, 0, 2).contiguous()
        recv = torch.empty_like(send)
        dist.all_to_all_single(recv, send, group=self.group)
        return recv.reshape(N * Br, Br)

    def forward(self, real, fake, h_fake, m_real, h_real, m_fake):
        flat = [real.reshape(self.B, -1), fake.reshape(self.B, -1)]
        if flat[0].shape[1] != self.K:
            raise ValueError(f"expected videos with {self.K} elements per sample, got {flat[0].shape[1]}")
        self.fake_shape = fake.shape
        if self.ctx_frames:
            self._ctx_backend(real, fake)
        self.dtypes = [t.dtype for t in (fake, h_fake, m_real, h_real, m_fake)]
        shift = self.be.cost_fwd(flat[0].contiguous(), flat[1].contiguous(), h_fake.contiguous(), m_real.contiguous(),
                                 h_real.contiguous(), m_fake.contiguous())
        self._allreduce(shift, dist.ReduceOp.MIN)               # one cost shift per problem for all ranks
        part = self.be.sinkhorn_fwd()
        self._allreduce(part, dist.ReduceOp.SUM)
        kscale = math.log2(math.e) / self.eps
        self.terms = part[:, 1] / kscale + shift * part[:, 0]   # xy, xx, yy
        self.loss = 2.0 * self.terms[0] - self.terms[1] - self.terms[2]        # gan_utils.py:225
        return self.loss, self.terms

    def _ctx_backend(self, real, fake):
        """(ctx_period, ctx_len) = (T*W*C, ctx_frames*W*C) of [B, H, T, W, C] videos; a backend for that hint"""
        for n, v in (("real", real), ("fake", fake)):
            if v.dim() != 5 or v.shape[0] != self.B or v.shape[2] != self.T:
                raise ValueError(f"{n}: ctx_frames > 0 needs [B, H, T, W, C] videos with B = {self.B}, T = {self.T}, "
                                 f"got shape {tuple(v.shape)}")
        if real.shape != fake.shape:
            raise ValueError(f"real {tuple(real.shape)} and fake {tuple(fake.shape)} differ in shape")
        frame = real.shape[3] * real.shape[4]
        ctx = (self.T * frame, self.ctx_frames * frame)
        if self.be is None or self.be.ctx != ctx:
            self.be = CudaMixedShardBackend(self.B, self.K, self.T, self.J, self.s, self.eps, self.L, self.row0,
                                            self.Brows, self.device, self.group, ctx=ctx)

    def backward(self, gloss=1.0):
        g3 = torch.tensor([2.0 * gloss, -gloss, -gloss], dtype=self.terms.dtype, device=self.terms.device)
        Cbar3 = self.be.sinkhorn_bwd(g3)
        XYcol = self._columns_of(Cbar3[0])
        YYcol = self._columns_of(Cbar3[2])
        g_fake, gh_fake, gm_real, gh_real, gm_fake = self.be.cost_bwd(XYcol, YYcol)
        self._allreduce(gm_real, dist.ReduceOp.SUM)
        self._allreduce(gm_fake, dist.ReduceOp.SUM)
        g_fake, gh_fake, gm_real, gh_real, gm_fake = _as_dtypes((g_fake, gh_fake, gm_real, gh_real, gm_fake), self.dtypes)
        return {"fake": g_fake.reshape((self.Brows,) + tuple(self.fake_shape[1:])), "h_fake": gh_fake, "m_real": gm_real,
                "h_real": gh_real, "m_fake": gm_fake}


def bench_cfg5(cx, cfg, K, config, steps, s, timed):
    """bench.py's config-5 leg on N > 1 ranks: one B = 8192 problem, rows sharded, strong scaling."""
    torch_ = cx.torch
    B, T = cfg["B"], cfg["T"]
    g = torch_.Generator(device=cx.dev).manual_seed(1)          # same seed on every rank: replicated inputs
    real = torch_.rand((B, K), generator=g, device=cx.dev)
    fake = torch_.rand((B, K), generator=g, device=cx.dev)
    hm = [torch_.sigmoid(torch_.randn((B, T, 8), generator=g, device=cx.dev)) for _ in range(4)]
    sm = ShardedMixedLoss(B, K, T, 8, s, device=cx.dev)
    lib = cx.lib
    n0 = lib.kccot_launch_count()

    def step(_i):
        sm.forward(real, fake, *hm)
        return sm.backward(1.0)
    grads = step(0)
    per_step = int(lib.kccot_launch_count() - n0)
    ms, clocks = timed(cx, step, steps, warmup=1)
    pk = {}
    try:
        import json
        import os
        with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")) as f:
            pk = json.load(f)
    except OSError:
        pass
    peak = float(pk.get("bf16_tflops_sustained", 1400.0)) * cx.world
    flops = 10.0 * B * B * K + 10.0 * B * B * (T - 1) * 8
    ach = flops / (ms * 1e-3 / steps) / 1e12
    nv = 2 * 100 * 3 * (B + 4) * 4 * (cx.world - 1)             # mailbox bytes sent per rank and evaluation
    out = {"value": steps / (ms * 1e-3), "unit": "evals/s", "steps": steps, "ms_per_step": ms / steps, "scaling": "strong",
           "config": config, "clocks": clocks, "gpu_launches_per_step": per_step,
           "parallelism": f"cost rows sharded over {cx.world} ranks ({B // cx.world} samples each), inputs replicated; "
                          "Sinkhorn column sums exchanged inside the persistent kernels (peer mailboxes over NVLink); NCCL: "
                          "MIN[3], SUM[6], 2 all-to-alls of [Brows,B], 2 SUM[B,T,J] per evaluation",
           "nvlink_bytes_per_rank_in_kernel": nv,
           "roofline": {"bound": "tensor", "scope": "whole step, all ranks", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                        "frac": ach / peak, "algorithmic_flops_per_step": flops,
                        "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained x ranks",
                        "note": "row shards cannot share the symmetric halves of the xx / yy blocks: 30 B^2 K executed "
                                "MMA flops per evaluation (3 fp16 products x (6 + 4) B^2 K)",
                        "executed_mma_frac": 30.0 * B * B * K / (ms * 1e-3 / steps) / 1e12 / peak, "traffic": None}}
    fin = bool(torch_.isfinite(sm.terms).all() and torch_.isfinite(grads["fake"]).all())
    out["parity"] = {"checked": True, "ok": fin, "finite": fin, "loss_terms": sm.terms.tolist(),
                     "against": "finiteness here; the sharded path is checked against the fp64 oracle at B = 1024 on 2 "
                                "ranks by tests/test_sharded_nccl.py (torchrun) and on CPU by tests/test_sharded_gloo.py"}
    return out
