"""Drop-in for `data_utils.KernelSmoothing` (neuripss2020/kccotgan, data_utils.py:478-586).

Only the kernel-smoothing class is on the loss hot path; the loaders, plotting helpers and LR
schedules of the reference's data_utils are out of scope (SURVEY.md §2).

The convolutions take CUDA fp32 or bf16 videos and return the input's dtype.  A bf16 video is smoothed by bf16
kernels with fp32 arithmetic inside: the output is the fp32 output on the widened video rounded to nearest even, and
the gradient is bf16 (kccot_smooth_fwd_bf16 / _bwd_bf16 in include/kccot.h).  Any other dtype raises ValueError.

`sigma` is a number, or a SmoothingTaps: a device buffer of weights that the kernels read when they run, so that a
CUDA graph captured with it follows an annealed sigma (the sigma changes between replays, the graph does not).

The *_batched convolutions smooth nprob independent videos [nprob, B, H, T, W, C] in one call, each with its own sigma
and divided by its own maximum: the result is that of nprob separate calls.
"""
import numbers

import numpy as np
import torch

from .functional import SmoothBatchedFn, SmoothFn, _check_video


class SmoothingTaps:
    """The 2r+1 Gaussian weights of one radius in a fixed-address device buffer, for the convolutions of a captured
    CUDA graph whose sigma changes between replays:

        taps = SmoothingTaps(ks.temporal_radius).set(5.0)
        (capture ks.temporal_convolution(x, taps) and its backward into a graph g)
        taps.set(ks.annealing_sigma(5.0, it)); g.replay()

    .set(sigma) writes KernelSmoothing._weights(radius, sigma), the host fp32 weights a float sigma uses, so the result
    is the float-sigma call's at the same sigma.  It is ordered on the current stream and does not synchronise the
    host (a pinned source copied with non_blocking=True).

    With `nprob`, the weights of nprob problems for the *_batched convolutions: `weights` is [nprob, 2r+1] and .set()
    takes one sigma for all of them or a sequence of nprob sigmas, row p holding KernelSmoothing._weights(radius,
    sigma_p)."""

    def __init__(self, radius, device="cuda", nprob=None):
        self.radius = int(radius)
        self.nprob = None if nprob is None else int(nprob)
        if self.nprob is not None and self.nprob < 1:
            raise ValueError(f"nprob must be at least 1, got {nprob}")
        shape = (2 * self.radius + 1,) if self.nprob is None else (self.nprob, 2 * self.radius + 1)
        self.weights = torch.zeros(shape, dtype=torch.float32, device=device)

    def set(self, sigma):
        if self.nprob is None:
            w = torch.from_numpy(KernelSmoothing._weights(self.radius, sigma))
        else:
            sig = [sigma] * self.nprob if isinstance(sigma, numbers.Real) else list(sigma)
            if len(sig) != self.nprob:
                raise ValueError(f"{len(sig)} sigmas for {self.nprob} problems")
            w = torch.from_numpy(np.stack([KernelSmoothing._weights(self.radius, s) for s in sig]))
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

    # -- batched independent problems ----------------------------------------------------------------
    def _batched(self, inputs, sigma, mode, radius):
        """checks as in the single-problem methods, then one SmoothBatchedFn call.  A number or sequence sigma becomes a
        SmoothingTaps whose weights are copied to the device on every call, which a CUDA graph cannot record."""
        if isinstance(sigma, SmoothingTaps):
            if sigma.radius != radius:
                raise ValueError(f"SmoothingTaps of radius {sigma.radius} for a filter of radius {radius}")
            nprob = inputs.shape[0] if isinstance(inputs, torch.Tensor) and inputs.dim() else None
            if sigma.nprob != nprob:
                raise ValueError(f"SmoothingTaps of {sigma.nprob} problems for a batch of {nprob} problems")
        inputs = _check_video(inputs, "inputs", 6)
        _, _, H, T, W, _ = inputs.shape
        for name, n in ((("T", T),) if mode == 1 else (("H", H), ("T", T), ("W", W))):
            self._check_axis(name, n, radius)
        if not isinstance(sigma, SmoothingTaps):
            if torch.cuda.is_current_stream_capturing():
                raise ValueError("a number or sequence sigma is copied to the device on every call, which CUDA graph "
                                 "capture cannot record: pass a SmoothingTaps(radius, nprob=...) and .set() it "
                                 "between replays")
            sigma = SmoothingTaps(radius, inputs.device, inputs.shape[0]).set(sigma)
        return SmoothBatchedFn.apply(inputs, mode, sigma)

    def temporal_convolution_batched(self, inputs, sigma):
        """temporal_convolution of nprob independent videos in one call: `inputs` [nprob, B, H, T, W, C] (fp32 or
        bf16), problem p filtered with sigma_p and divided by its own maximum.  `sigma`: a number, a sequence of nprob
        numbers, or a SmoothingTaps(temporal_radius, nprob=nprob)."""
        return self._batched(inputs, sigma, 1, self.temporal_radius)

    def gaussian_convolution3D_batched(self, inputs, sigma):
        """gaussian_convolution3D of nprob independent videos in one call: `inputs` [nprob, B, H, T, W, C] (fp32 or
        bf16), problem p filtered with sigma_p and divided by its own maximum.  `sigma`: a number, a sequence of nprob
        numbers, or a SmoothingTaps(spatial_radius, nprob=nprob)."""
        return self._batched(inputs, sigma, 3, self.spatial_radius)

    def annealing_sigma(self, init_sigma, step, decay_steps=500, decay_rate=0.975):
        """data_utils.py:584-586."""
        return init_sigma * decay_rate ** (step / decay_steps)
