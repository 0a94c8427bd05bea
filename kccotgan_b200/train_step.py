"""The two step closures of the reference's training loop (kernel_train.py:219-292) around the B200 loss
path, with STUB networks (SURVEY.md §8 f2).

The generator (ConvLSTM encoder/decoder) and the two discriminators of the reference are out of scope; the
stubs below only produce tensors of the right shapes and ranges — `fake_pred` in the sigmoid range
[B,H,pred,W,C] (gan.py:358-360) and `[B,T,J]` sigmoid features (gan.py:418) — so that one
`kernel_train.py` iteration (discriminator step + generator step, optional kernel smoothing, both Adam
updates) can be run and timed end to end with the loss path in place.  The order of operations, the loss
formulas (`disc_loss = -loss + pM`, generator loss = `loss`) and the argument orders follow the reference
line by line.
"""
import torch
from torch import nn

from . import gan_utils
from .data_utils import KernelSmoothing, SmoothingTaps


class StubGenerator(nn.Module):
    """real_in [B,H,ctx,W,C] + noise -> fake_pred [B,H,pred,W,C] in (0,1).  A per-pixel affine map of the
    last context frame plus a learned per-step offset driven by the noise: cheap, differentiable, and every
    parameter receives a gradient from the loss."""

    def __init__(self, pred_steps, channels, z_dim=8):
        super().__init__()
        self.pred_steps = pred_steps
        self.gain = nn.Parameter(torch.ones(pred_steps, 1, channels))
        self.bias = nn.Parameter(torch.zeros(pred_steps, 1, channels))
        self.z_proj = nn.Linear(z_dim, pred_steps * channels)
        self.z_dim = z_dim

    def forward(self, real_in, z):
        B, H, _, W, C = real_in.shape
        last = real_in[:, :, -1:, :, :]                                    # [B,H,1,W,C]
        zc = self.z_proj(z).reshape(B, 1, self.pred_steps, 1, C)           # [B,1,pred,1,C]
        logits = 4.0 * (last - 0.5) * self.gain + self.bias + zc
        return torch.sigmoid(logits)


class StubDiscriminator(nn.Module):
    """video [B,H,T,W,C] -> [B,T,J] in (0,1): frame-wise linear features followed by a causal running mean
    (stands in for the LSTM stack of gan.py:411-429: output t depends on frames <= t only).

    The spatial pooling is a mean over a strided VIEW of the video as it lies in memory ([B,H/p,p,T,W/p,p,C]): no
    transposed copy of the 31 MB tensor and a broadcast for a backward (a permute + AvgPool2d version spent 0.9 ms of
    a 2.1 ms training iteration in the permute copies and avg_pool2d_backward)."""

    def __init__(self, height, width, channels, J=8, pool=8):
        super().__init__()
        self.p = pool
        self.lin = nn.Linear((height // pool) * (width // pool) * channels, J)

    def forward(self, video):
        B, H, T, W, C = video.shape
        p = self.p
        pooled = video.reshape(B, H // p, p, T, W // p, p, C).mean(dim=(2, 5))          # [B,H/p,T,W/p,C]
        feat = self.lin(pooled.permute(0, 2, 1, 3, 4).reshape(B * T, -1)).reshape(B, T, -1)
        steps = torch.arange(1, T + 1, device=video.device, dtype=video.dtype).reshape(1, T, 1)
        return torch.sigmoid(torch.cumsum(feat, dim=1) / steps)


def _kernel_smoothing():
    return KernelSmoothing(temporal_kernel_size=6, spatial_kernel_size=6)                  # kernel_train.py:216


def make_training_steps(generator, discriminator_h, discriminator_m, batch_size, scaling_coef=1.0 / 15.0,
                        sinkhorn_eps=0.8, sinkhorn_l=100, reg_penalty=1.0, kernel_choice="none", gen_lr=1e-4,
                        disc_lr=1e-4, seed=1, capturable=False):
    """Returns (disc_training_step, gen_training_step), each `(real_in, real_pred, sigma) -> scalar tensor`,
    mirroring kernel_train.py:219-292 (Adam with beta_1 = 0.5, beta_2 = 0.9 as at :62-63; the LR schedule is the caller's).
    `sigma` is a number or a data_utils.SmoothingTaps of the smoothing's radius (3)."""
    # capturable=True: the variant GraphedTrainingIteration records into a CUDA graph (Adam keeps its step count on
    # the device, the noise comes from the default CUDA generator, which graphs know how to advance)
    gen_opt = torch.optim.Adam(generator.parameters(), lr=gen_lr, betas=(0.5, 0.9), capturable=capturable)
    dischm_opt = torch.optim.Adam(list(discriminator_h.parameters()) + list(discriminator_m.parameters()), lr=disc_lr,
                                  betas=(0.5, 0.9), capturable=capturable)
    gaussian_kernel = _kernel_smoothing()
    dev = next(generator.parameters()).device
    noise = torch.Generator(device=dev)
    noise.manual_seed(seed)

    def _forward(real_in, real_pred, sigma):
        hidden_z = torch.randn((batch_size, generator.z_dim), generator=None if capturable else noise, device=dev)   # :221 / :257
        fake_pred = generator(real_in, hidden_z)
        real = torch.cat((real_in, real_pred), dim=2)                                          # :227 / :264
        fake = torch.cat((real_in, fake_pred), dim=2)                                          # :228 / :265
        if kernel_choice == "1d":                                                              # :230-232
            real = gaussian_kernel.temporal_convolution(real, sigma)
            fake = gaussian_kernel.temporal_convolution(fake, sigma)
        elif kernel_choice == "2d":                                                            # :234-236 (raises)
            real = gaussian_kernel.spatial_convolution(real, sigma)
            fake = gaussian_kernel.spatial_convolution(fake, sigma)
        elif kernel_choice == "3d":                                                            # :238-240
            real = gaussian_kernel.gaussian_convolution3D(real, sigma)
            fake = gaussian_kernel.gaussian_convolution3D(fake, sigma)
        h_fake = discriminator_h(fake)                                                         # :242-246
        h_real = discriminator_h(real)
        m_real = discriminator_m(real)
        m_fake = discriminator_m(fake)
        loss = gan_utils.compute_sinkhorn_loss(real, fake, scaling_coef, sinkhorn_eps, sinkhorn_l, h_fake, m_real,
                                               h_real, m_fake, video=True)                     # :247
        return loss, m_real

    def disc_training_step(real_in, real_pred, sigma):
        loss, m_real = _forward(real_in, real_pred, sigma)
        pm1 = gan_utils.scale_invariante_martingale_regularization(m_real, reg_penalty, scaling_coef)   # :249
        disc_loss = -loss + pm1                                                                # :250
        dischm_opt.zero_grad(set_to_none=True)
        generator.zero_grad(set_to_none=True)
        disc_loss.backward()                                                                   # :252-253
        dischm_opt.step()                                                                      # :254-255
        return pm1.detach()

    def gen_training_step(real_in, real_pred, sigma):
        loss, _ = _forward(real_in, real_pred, sigma)
        gen_opt.zero_grad(set_to_none=True)
        discriminator_h.zero_grad(set_to_none=True)
        discriminator_m.zero_grad(set_to_none=True)
        loss.backward()                                                                        # :289
        gen_opt.step()                                                                         # :290-291
        return loss.detach()

    return disc_training_step, gen_training_step


class GraphedTrainingIteration:
    """One kernel_train.py iteration — discriminator step, then generator step (kernel_train.py:300-310) — recorded
    ONCE into a CUDA graph and replayed with a single launch: with the loss path at ~0.13 ms per evaluation the eager
    iteration is dominated by the ~150 small launches of the networks and optimisers around it.

        it = GraphedTrainingIteration(gen, disc_h, disc_m, real_in_example, real_pred_example)
        it.real_in.copy_(x[:, :, :ctx]); it.real_pred.copy_(x[:, :, ctx:])
        loss, pm = it.step()                   # or it.step(sigma), e.g. sigma = annealing_sigma(init_sig, iteration)

    Static-buffer contract as in graphed.GraphedSinkhornLoss.  With `kernel_choice` "1d" / "3d" the smoothing reads its
    weights from a data_utils.SmoothingTaps captured with the graph: step(sigma) writes the weights of `sigma` there
    before the replay (kernel_train.py's annealed sigma, :308-311), and step() replays the constructor's `sigma`."""

    def __init__(self, generator, discriminator_h, discriminator_m, real_in, real_pred, sigma=5.0, warmup=3, **kw):
        self.real_in = real_in.detach().clone()
        self.real_pred = real_pred.detach().clone()
        dev = self.real_in.device
        self._disc, self._gen = make_training_steps(generator, discriminator_h, discriminator_m, real_in.shape[0],
                                                    capturable=True, **kw)
        self.sigma = self._sigma_set = sigma
        self.taps = None
        kernel_choice = kw.get("kernel_choice", "none")
        if kernel_choice in ("1d", "3d"):
            ks = _kernel_smoothing()
            self.taps = SmoothingTaps(ks.temporal_radius if kernel_choice == "1d" else ks.spatial_radius,
                                      device=dev).set(sigma)
            sigma = self.taps
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                    # optimiser state and library attributes come to life here
            for _ in range(max(1, warmup)):
                self._disc(self.real_in, self.real_pred, sigma)
                self._gen(self.real_in, self.real_pred, sigma)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.pm = self._disc(self.real_in, self.real_pred, sigma)
            self.loss = self._gen(self.real_in, self.real_pred, sigma)

    def step(self, sigma=None):
        """One replay at `sigma` (None: the constructor's); without smoothing sigma is unused, as in the eager steps."""
        sigma = self.sigma if sigma is None else sigma
        if self.taps is not None and sigma != self._sigma_set:
            self.taps.set(sigma)
            self._sigma_set = sigma
        self.graph.replay()
        return self.loss, self.pm
