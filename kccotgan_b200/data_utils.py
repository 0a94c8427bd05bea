"""Drop-in for `data_utils.KernelSmoothing` (neuripss2020/kccotgan, data_utils.py:478-586).

Only the kernel-smoothing class is on the loss hot path; the loaders, plotting helpers and LR
schedules of the reference's data_utils are out of scope (SURVEY.md §2).

The convolutions take CUDA fp32 or bf16 videos and return the input's dtype.  A bf16 video is smoothed by bf16
kernels with fp32 arithmetic inside: the output is the fp32 output on the widened video rounded to nearest even, and
the gradient is bf16 (kccot_smooth_fwd_bf16 / _bwd_bf16 in include/kccot.h).  Any other dtype raises ValueError.

`sigma` is a number, or a SmoothingTaps: a device buffer of weights that the kernels read when they run, so that a
CUDA graph captured with it follows an annealed sigma (the sigma changes between replays, the graph does not).
"""
import numpy as np
import torch

from .functional import SmoothFn, _check_video


class SmoothingTaps:
    """The 2r+1 Gaussian weights of one radius in a fixed-address device buffer, for the convolutions of a captured
    CUDA graph whose sigma changes between replays:

        taps = SmoothingTaps(ks.temporal_radius).set(5.0)
        (capture ks.temporal_convolution(x, taps) and its backward into a graph g)
        taps.set(ks.annealing_sigma(5.0, it)); g.replay()

    .set(sigma) writes KernelSmoothing._weights(radius, sigma), the host fp32 weights a float sigma uses, so the result
    is the float-sigma call's at the same sigma.  It is ordered on the current stream and does not synchronise the
    host (a pinned source copied with non_blocking=True)."""

    def __init__(self, radius, device="cuda"):
        self.radius = int(radius)
        self.weights = torch.zeros(2 * self.radius + 1, dtype=torch.float32, device=device)

    def set(self, sigma):
        w = torch.from_numpy(KernelSmoothing._weights(self.radius, sigma))
        self.weights.copy_(w.pin_memory() if self.weights.is_cuda else w, non_blocking=True)
        return self


class KernelSmoothing:
    """Gaussian smoothing of [B,H,T,W,C] videos, divided by the global max of the result."""

    def __init__(self, temporal_kernel_size=6, spatial_kernel_size=8):
        # data_utils.py:479-481
        self.temporal_radius = temporal_kernel_size // 2
        self.spatial_radius = spatial_kernel_size // 2

    # -- weights --------------------------------------------------------------------------------
    @staticmethod
    def _weights(radius, sigma):
        """fp32 arithmetic exactly as data_utils.py:487-490."""
        sigma2 = np.float32(sigma) * np.float32(sigma)
        x = np.arange(-radius, radius + 1, dtype=np.float32)
        k = np.exp((np.float32(-0.5) / sigma2) * x ** 2, dtype=np.float32)
        return (k / k.sum(dtype=np.float32)).astype(np.float32)

    def gaussian_kernel1d(self, radius, sigma, device="cuda"):
        """data_utils.py:483-491 — [2r+1] normalised Gaussian weights."""
        return torch.from_numpy(self._weights(radius, sigma)).to(device)

    def gaussian_kernel3d(self, radius, sigma, device="cuda"):
        """data_utils.py:493-501 — [2r+1,2r+1,2r+1,1,1]; equals w (x) w (x) w up to fp32 rounding."""
        x = np.arange(-radius, radius + 1, dtype=np.float32)
        xx, yy, zz = np.meshgrid(x, x, x)
        sigma2 = np.float32(sigma) * np.float32(sigma)
        k = np.exp((np.float32(-0.5) / sigma2) * (xx ** 2 + yy ** 2 + zz ** 2), dtype=np.float32)
        k = (k / k.sum(dtype=np.float32)).astype(np.float32)
        return torch.from_numpy(k[:, :, :, None, None]).to(device)

    # -- convolutions ---------------------------------------------------------------------------
    @staticmethod
    def _check_axis(name, n, radius):
        if n <= radius:
            raise ValueError(f"REFLECT padding by {radius} needs the {name} axis longer than {radius}, got {n}")

    @staticmethod
    def _taps(radius, sigma):
        """the weights SmoothFn takes: a SmoothingTaps of this radius, or the host weights of a number"""
        if isinstance(sigma, SmoothingTaps):
            if sigma.radius != radius:
                raise ValueError(f"SmoothingTaps of radius {sigma.radius} for a filter of radius {radius}")
            return sigma
        return tuple(KernelSmoothing._weights(radius, sigma))

    def temporal_convolution(self, inputs, sigma):
        """data_utils.py:503-521 — (2r+1)-tap REFLECT filter along T, / global max.  `sigma`: a number or a
        SmoothingTaps of radius temporal_radius."""
        taps = self._taps(self.temporal_radius, sigma)
        inputs = _check_video(inputs, "inputs", 5)
        self._check_axis("T", inputs.shape[2], self.temporal_radius)
        return SmoothFn.apply(inputs, 1, taps, None)

    def spatial_convolution(self, inputs, sigma):
        """data_utils.py:523-550 — BROKEN in the reference: the VALID conv2d shrinks H, W by 2r and the
        following reshape to the original [.., h, w] fails (:537-538, :547-548).  Reproduced as an error."""
        bs, h, t, w, nc = inputs.shape
        r = self.spatial_radius
        raise ValueError(f"spatial_convolution: cannot reshape the VALID-convolved tensor of "
                         f"{bs * nc * t * (h - 2 * r) * (w - 2 * r)} elements into {[bs, nc, t, h, w]} "
                         "(the reference's '2d' kernel raises here, data_utils.py:537-538)")

    def gaussian_convolution3D(self, inputs, sigma):
        """data_utils.py:552-582 — (2r+1)^3 REFLECT filter over (H,T,W) per channel (three separable
        passes), / global max.  Uses the SPATIAL radius for all three axes (:553,562-564).  `sigma`: a number or a
        SmoothingTaps of radius spatial_radius."""
        taps = self._taps(self.spatial_radius, sigma)
        inputs = _check_video(inputs, "inputs", 5)
        _, H, T, W, _ = inputs.shape
        for name, n in (("H", H), ("T", T), ("W", W)):
            self._check_axis(name, n, self.spatial_radius)
        return SmoothFn.apply(inputs, 3, None, taps)

    def annealing_sigma(self, init_sigma, step, decay_steps=500, decay_rate=0.975):
        """data_utils.py:584-586."""
        return init_sigma * decay_rate ** (step / decay_steps)
