"""Drop-in for the reference's `gan_utils` module (neuripss2020/kccotgan, gan_utils.py).

Same function names, positional orders and defaults; inputs are torch CUDA fp32 tensors instead of
TensorFlow eager tensors, outputs are tensors on the autograd tape (0-d where the reference
returns a scalar).  All arithmetic runs in libkccot's sm_100a kernels (include/kccot.h).
The mixed loss (compute_sinkhorn_loss and its variants below) also takes bf16 videos: the result is
exactly that of the fp32 call on the widened videos, the video gradients come back in bf16 (the fp32
gradient rounded to nearest even), and two bf16 videos are read as bf16 by the kernels (no fp32 copy
at B <= 64 with B % 8 == 0 and K % 8 == 0, K >= 128).  So can a bf16 video smoothed first by
data_utils.KernelSmoothing, which returns bf16 (the whole smoothing -> loss -> adjoints chain then makes no fp32
copy of a video).  scale_invariante_martingale_regularization_batched widens a bf16 M (exact) and returns its gradient
in bf16.  The other functions here stay fp32-only.

Reference quirks are reproduced on purpose (SURVEY.md Appendix B):
  * compute_sinkhorn_loss passes `sinkhorn_eps, sinkhorn_l` positionally into compute_sinkhorn's
    `hx, My` slots (gan_utils.py:221-223 vs :124), so the mixed loss ALWAYS solves with
    epsilon=1.0, L=100;
  * the martingale term indexes h by the ROW sample and Delta M by the COLUMN sample (:34-38);
  * Lmin = 100 is hard-coded in compute_sinkhorn (:149): with L <= 100 there is no early exit;
  * the returned cost is the sharp sum(pi * C) and the gradient is the fully unrolled one.
"""
import torch

from .functional import (CostFn, MartingalePenaltyBatchedFn, MartingalePenaltyFn, MixedLossBatchedFn, MixedLossFn,
                         SinkhornFn, _check_video)

__all__ = ["cost_xy", "modified_cost", "bi_causal_modified_cost", "benchmark_sinkhorn", "compute_sinkhorn",
           "compute_N", "scale_invariante_martingale_regularization", "compute_sinkhorn_loss"]


def cost_xy(x, y, scaling_coef):
    """gan_utils.py:6-18 — [B,T,D] x [B,T,D] -> [B,B], s * sum_{t,d} (x_i - y_j)^2."""
    return CostFn.apply(x, y, None, None, None, None, scaling_coef)


def modified_cost(x, y, h, M, scaling_coef):
    """gan_utils.py:21-43 — cost_xy + s * sum_{t<T-1} h[i,t] . (M[j,t+1] - M[j,t])."""
    return CostFn.apply(x, y, h, M, None, None, scaling_coef)


def bi_causal_modified_cost(x, y, hy, Mx, hx, My, scaling_coef):
    """gan_utils.py:46-72 — modified_cost plus the second s * hx[i] . Delta My[j] term."""
    return CostFn.apply(x, y, hy, Mx, hx, My, scaling_coef)


def benchmark_sinkhorn(x, y, scaling_coef, epsilon=1.0, L=10, Lmin=10):
    """gan_utils.py:75-121 — non-causal Sinkhorn on cost_xy; stops after iteration index i >= Lmin
    once sum|u - u_prev| < 1e-2 (:116).  The test runs on the device."""
    C = cost_xy(x, y, scaling_coef)
    cost, _ = SinkhornFn.apply(C.unsqueeze(0), epsilon, L, Lmin, 1e-2, True)
    return cost[0]


def compute_sinkhorn(x, y, hy, Mx, scaling_coef, hx=None, My=None, epsilon=1.0, L=100, bi_causal=False):
    """gan_utils.py:124-165 — causal Sinkhorn cost sum(pi * C) after L log-domain iterations
    (stops early only if L > 100 and sum|u - u_prev| < 1e-2 after >= 100 iterations)."""
    if bi_causal:
        C = bi_causal_modified_cost(x, y, hy, Mx, hx, My, scaling_coef)
    else:
        C = modified_cost(x, y, hy, Mx, scaling_coef)
    cost, _ = SinkhornFn.apply(C.unsqueeze(0), epsilon, L, 100, 1e-2, False)
    return cost[0]


def compute_N(M):
    """gan_utils.py:168-176 — first difference along axis 1 of a [batch, T] tensor (unused by the
    training loop; pure indexing, no kernel needed)."""
    T = M.shape[1]
    return M[:, 1:] - M[:, :T - 1]


def scale_invariante_martingale_regularization(M, reg_lam, scaling_coef):
    """gan_utils.py:179-201 — p_M."""
    return MartingalePenaltyFn.apply(M, reg_lam, scaling_coef)


def scale_invariante_martingale_regularization_batched(M, reg_lam, scaling_coef):
    """Not in the reference: p_M of `nprob` independent problems in one call (BASELINE config 4's discriminator step,
    kernel_train.py:249-250).  M is [nprob, B, T, J], fp32 or bf16; returns the [nprob] penalties, entry p bit-identical
    to scale_invariante_martingale_regularization(M[p].float(), ...) and differentiable w.r.t. M[p] only.  Folding the
    problems into the batch axis would not do: the mean, sigma_j and A_tj are taken over the batch."""
    return MartingalePenaltyBatchedFn.apply(M, reg_lam, scaling_coef)


def compute_sinkhorn_loss(f_real, f_fake, scaling_coef, sinkhorn_eps, sinkhorn_l, h_fake, m_real, h_real,
                          m_fake, video=True):
    """gan_utils.py:204-227 — 2*S(real,fake; h_fake,m_real) - S(real,real; h_real,m_real)
    - S(fake,fake; h_fake,m_fake).

    `sinkhorn_eps` and `sinkhorn_l` are accepted and IGNORED exactly as in the reference (they land
    in compute_sinkhorn's unused `hx`/`My` parameters): epsilon=1.0, L=100 always.
    video=True: f_* are [B,H,T,W,C]; the reference's transpose to [B,T,HWC] (:217-220) only
    permutes axes that the cost sums over, so the tensors are consumed in place as [B, K].
    video=False: f_* are [B,T,D].  One fused pass: the three cost matrices come from a single
    stacked Gram of [real; fake], the three solves run as three CTAs of one launch.
    """
    del sinkhorn_eps, sinkhorn_l      # reference quirk, see module docstring
    f_real = _check_video(f_real, "f_real")
    f_fake = _check_video(f_fake, "f_fake")
    if video and (f_real.dim() != 5 or f_fake.dim() != 5):
        raise ValueError(f"video=True expects [B,H,T,W,C] tensors, got {tuple(f_real.shape)} / {tuple(f_fake.shape)}")
    if not video and (f_real.dim() != 3 or f_fake.dim() != 3):
        raise ValueError(f"video=False expects [B,T,D] tensors, got {tuple(f_real.shape)} / {tuple(f_fake.shape)}")
    loss, _ = MixedLossFn.apply(f_real, f_fake, h_fake, m_real, h_real, m_fake, scaling_coef, 1.0, 100)
    return loss


def sinkhorn_loss_terms(f_real, f_fake, scaling_coef, h_fake, m_real, h_real, m_fake, epsilon=1.0, L=100):
    """Not in the reference: the same fused solve, returning (loss, [loss_xy, loss_xx, loss_yy]) and
    honouring epsilon / L (what the reference's CLI flags were meant to control)."""
    return MixedLossFn.apply(f_real, f_fake, h_fake, m_real, h_real, m_fake, scaling_coef, epsilon, L)


def compute_sinkhorn_loss_shared_context(f_real, f_fake, scaling_coef, h_fake, m_real, h_real, m_fake, ctx_frames,
                                         epsilon=1.0, L=100):
    """Not in the reference's API, but in its data flow: kernel_train.py:225-226 / :267-268 build
    real = concat(real_in, real_pred) and fake = concat(real_in, fake_pred) along the time axis, so with
    `--kernel none` the first `ctx_frames` frames of the two [B,H,T,W,C] videos are the same numbers.  Stating that
    lets the kernels skip them: the forward never reads fake's context frames (bit-identical loss), the backward
    neither reads nor computes the gradient of fake's context frames — they are constants (copies of the data), and
    the returned gradient is ZERO there instead of the value the reference's tape would hand to the data tensor.
    Saves ctx/T of the fake video's forward traffic and ctx/T of the whole backward.  Not valid after temporal or
    3-D smoothing (it leaks predicted frames into the context frames).  Returns (loss, [xy, xx, yy])."""
    f_real = _check_video(f_real, "f_real")
    f_fake = _check_video(f_fake, "f_fake")
    if f_real.dim() != 5 or f_fake.dim() != 5:
        raise ValueError(f"expected [B,H,T,W,C] videos, got {tuple(f_real.shape)} / {tuple(f_fake.shape)}")
    T, W, C = f_real.shape[2], f_real.shape[3], f_real.shape[4]
    ctx_frames = int(ctx_frames)
    if not 0 <= ctx_frames < T:
        raise ValueError(f"ctx_frames must be in [0, T) = [0, {T}), got {ctx_frames}")
    return MixedLossFn.apply(f_real, f_fake, h_fake, m_real, h_real, m_fake, scaling_coef, epsilon, L,
                             (T * W * C, ctx_frames * W * C))


def compute_sinkhorn_loss_batched(f_real, f_fake, scaling_coef, h_fake, m_real, h_real, m_fake, epsilon=1.0, L=100):
    """Not in the reference: `nprob` independent (real, fake, h, m) tuples in one call (BASELINE config 4:
    "batched independent Sinkhorn problems").  Every tensor carries a leading problem axis
    (f_* [nprob,B,...], h/m [nprob,B,T,J]); returns the [nprob] mixed losses of gan_utils.py:204-227, each
    differentiable w.r.t. its own inputs.  Problems share nothing, so ranks can split them with no collective."""
    loss, _ = MixedLossBatchedFn.apply(f_real, f_fake, h_fake, m_real, h_real, m_fake, scaling_coef, epsilon, L)
    return loss
