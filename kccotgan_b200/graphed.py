"""CUDA-graph replay of the loss forward+backward (launch-bound inner loop → one graph launch).

The eager entry point (`gan_utils.compute_sinkhorn_loss` + autograd) issues ~10 kernels from Python per
evaluation; at B=64 the kernels take ~200 us and the launch gaps another ~70 us.  `GraphedSinkhornLoss`
captures the same C-ABI launch chain once on static buffers and replays it with a single
`cudaGraphLaunch`.  Contract (the usual static-buffer one): the caller writes the step's tensors into
`.real, .fake, .h_fake, .m_real, .h_real, .m_fake` (or passes tensors that already live there), calls
`step()`, and reads `.loss` and `.grads[...]`; no host synchronisation is involved.  `real` and `fake` may both be
bf16 (the gradients of the videos are then bf16 too); h / m are fp32.
"""
import torch

from . import gan_utils

_NAMES = ("real", "fake", "h_fake", "m_real", "h_real", "m_fake")


class GraphedSinkhornLoss:
    def __init__(self, real, fake, h_fake, m_real, h_real, m_fake, scaling_coef, want_real_grad=False,
                 adopt=True, warmup=2, ctx_frames=0):
        """Captures compute_sinkhorn_loss(...) and its gradients w.r.t. fake, h_fake, m_real, h_real,
        m_fake (and real if asked).  adopt=True uses the given tensors themselves as the static buffers
        (zero copies: later steps must overwrite them in place); adopt=False clones them."""
        srcs = (real, fake, h_fake, m_real, h_real, m_fake)
        for t, n in zip(srcs, _NAMES):
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype in (torch.float32, torch.bfloat16)):
                raise ValueError(f"{n}: expected a CUDA float32 tensor")
        # bf16 videos (the bf16 entry points of the library) when both are bf16; h / m stay fp32
        if real.dtype != fake.dtype or any(t.dtype != torch.float32 for t in srcs[2:]):
            raise ValueError("real / fake: expected both float32 or both bfloat16; h / m: expected float32")
        self.scaling_coef = float(scaling_coef)
        self.ctx_frames = int(ctx_frames)       # > 0: gan_utils.compute_sinkhorn_loss_shared_context
        bufs = [t.detach() if adopt else t.detach().clone() for t in srcs]
        bufs = [b.contiguous() for b in bufs]
        for b, n in zip(bufs, _NAMES):
            b.requires_grad_(n != "real" or want_real_grad)
            setattr(self, n, b)
        self._leaves = [b for b in bufs if b.requires_grad]
        self._leaf_names = [n for b, n in zip(bufs, _NAMES) if b.requires_grad]
        dev = bufs[0].device
        self._one = torch.ones((), dtype=torch.float32, device=dev)   # static gradient seed (no fill kernel per step)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                     # warm-up outside capture (attribute setting, caches)
            for _ in range(max(1, warmup)):
                self._eager()
        torch.cuda.current_stream(dev).wait_stream(side)
        from . import _lib
        n0 = _lib.load().kccot_launch_count()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss, g = self._eager()
            self.grads = dict(zip(self._leaf_names, g))
        self.kernels_per_replay = int(_lib.load().kccot_launch_count() - n0)   # libkccot kernels in the graph

    def _eager(self):
        if self.ctx_frames > 0:
            loss, _ = gan_utils.compute_sinkhorn_loss_shared_context(self.real, self.fake, self.scaling_coef,
                                                                     self.h_fake, self.m_real, self.h_real,
                                                                     self.m_fake, self.ctx_frames)
        else:
            loss = gan_utils.compute_sinkhorn_loss(self.real, self.fake, self.scaling_coef, 0.8, 100, self.h_fake,
                                                   self.m_real, self.h_real, self.m_fake, video=self.real.dim() == 5)
        return loss, torch.autograd.grad(loss, self._leaves, grad_outputs=self._one)

    def step(self):
        """Replay: recomputes .loss and .grads from the current contents of the static inputs."""
        self.graph.replay()
        return self.loss


class EvaluationLanes:
    """Independent evaluations in flight at once, one CUDA stream ("lane") per evaluator.

    One evaluation at B <= 64 is a chain of six kernels of which the two Sinkhorn kernels occupy 3 of the 148 SMs
    for ~40 % of the time, and every HBM kernel pays a few microseconds of ramp and prologue.  Evaluations that do not
    depend on each other (micro-batches, data-parallel replicas that share a GPU, the problems of BASELINE config 4,
    the discriminator- and generator-step losses of different batches) can be replayed on separate streams: the
    Sinkhorn kernels of one hide under the HBM kernels of the others.  Results are bit-identical to serial replays
    (each evaluator owns its buffers; nothing is shared between lanes).

        lanes = EvaluationLanes([GraphedSinkhornLoss(...), GraphedSinkhornLoss(...), ...])
        lanes.fork()                       # lanes wait for what the current stream has queued (input writes)
        for j in range(len(lanes)): lanes.submit(j)
        lanes.join()                       # the current stream waits for every lane
    """

    def __init__(self, evaluators, n_lanes=None):
        """evaluator j replays on stream j % n_lanes (default: one stream per evaluator)."""
        if not evaluators:
            raise ValueError("EvaluationLanes needs at least one evaluator")
        self.evaluators = list(evaluators)
        n_lanes = len(self.evaluators) if n_lanes is None else int(n_lanes)
        if n_lanes < 1:
            raise ValueError("n_lanes must be >= 1")
        dev = self.evaluators[0].real.device
        self.device = dev
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(min(n_lanes, len(self.evaluators)))]

    def __len__(self):
        return len(self.evaluators)

    def fork(self):
        cur = torch.cuda.current_stream(self.device)
        for s in self.streams:
            s.wait_stream(cur)

    def submit(self, j):
        """Replays evaluator j on its lane's stream; returns the evaluator (read .loss / .grads after join())."""
        ev = self.evaluators[j]
        with torch.cuda.stream(self.streams[j % len(self.streams)]):
            ev.graph.replay()
        return ev

    def join(self):
        cur = torch.cuda.current_stream(self.device)
        for s in self.streams:
            cur.wait_stream(s)
