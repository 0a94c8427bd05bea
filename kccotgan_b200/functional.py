"""torch.autograd glue between the reference-shaped Python functions and the C ABI.

PyTorch supplies device memory, streams and the tape only; every arithmetic step is a libkccot
kernel.  Tensors must be CUDA fp32 — anything else raises ValueError (no fallback) — except in the mixed loss
(MixedLossFn, MixedLossBatchedFn), which also takes bf16 videos and h / m: two bf16 videos run the bf16 entry points
of the library (the result is exactly the fp32 one on the widened videos, video gradients rounded to bf16); a bf16
video next to an fp32 one, and bf16 h / m, are widened with .float() (exact).  Gradients come back in the dtype of
their input.  The smoothing (SmoothFn) also takes bf16 videos: they run the bf16 entry points, whose output is the
fp32 output on the widened video rounded to bf16, and whose gradient is bf16 (see kccot_smooth_fwd_bf16 in kccot.h).
SmoothBatchedFn smooths nprob independent videos in one call, in fp32 or bf16 alike.  MartingalePenaltyBatchedFn
computes nprob independent penalties in one call; a bf16 M is widened with .float() (exact) and its gradient comes back
in bf16.
"""
import ctypes

import torch

from . import _lib

# default kernel-path flag; tests flip it through `set_path` to cross-check tcgen05 vs CUDA cores
_PATH = {"flags": _lib.PATH_AUTO}


def set_path(name):
    """'auto' | 'simt' | 'tcgen05' — which kernel family the cost GEMMs use (tests only)."""
    _PATH["flags"] = {"auto": _lib.PATH_AUTO, "simt": _lib.PATH_SIMT, "tcgen05": _lib.PATH_TCGEN05}[name]


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream(dev):
    # raw handle of the current stream of `dev` (torch.cuda.current_stream(dev).cuda_stream costs ~10 us per call)
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(dev.index if dev.index is not None else torch.cuda.current_device()))


class _on_device:
    """`with torch.cuda.device(dev)` only when `dev` is not already the current device (the common case costs one
    query instead of two device switches)."""
    __slots__ = ("dev", "ctx")

    def __init__(self, dev):
        self.dev = dev
        self.ctx = None

    def __enter__(self):
        idx = self.dev.index
        if idx is not None and idx != torch._C._cuda_getDevice():
            self.ctx = torch.cuda.device(self.dev)
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
        return False


def _check(t, name, ndim=None):
    if not isinstance(t, torch.Tensor):
        raise ValueError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (kccotgan_b200 has no CPU path), got {t.device}")
    if t.dtype != torch.float32:
        raise ValueError(f"{name}: expected float32, got {t.dtype}")
    if ndim is not None and t.dim() != ndim:
        raise ValueError(f"{name}: expected {ndim} dimensions, got shape {tuple(t.shape)}")
    return t.contiguous()


def _check_video(t, name, ndim=None):
    """A CUDA video of the mixed loss or the smoothing: fp32 or bf16, made contiguous."""
    if isinstance(t, torch.Tensor) and t.dtype == torch.bfloat16:
        if not t.is_cuda:
            raise ValueError(f"{name}: expected a CUDA tensor (kccotgan_b200 has no CPU path), got {t.device}")
        if ndim is not None and t.dim() != ndim:
            raise ValueError(f"{name}: expected {ndim} dimensions, got shape {tuple(t.shape)}")
        return t.contiguous()
    return _check(t, name, ndim)


def _videos(real, fake):
    """-> (real, fake, bf16).  Two bf16 videos stay bf16 (cloned if a view is not 16-byte aligned, as the bf16 entry
    points require); otherwise a bf16 one is widened to fp32, which is exact."""
    real, fake = _check_video(real, "f_real"), _check_video(fake, "f_fake")
    if real.dtype == fake.dtype == torch.bfloat16:
        return (real if real.data_ptr() % 16 == 0 else real.clone(),
                fake if fake.data_ptr() % 16 == 0 else fake.clone(), True)
    return real.float(), fake.float(), False


def _check_hm(t, name, ndim):
    """h / m of the mixed loss: fp32, or bf16 widened to fp32 (exact)."""
    if isinstance(t, torch.Tensor) and t.dtype == torch.bfloat16:
        t = t.float()
    return _check(t, name, ndim)


def _as_dtypes(grads, dtypes):
    """each gradient in the dtype of its input (the fp32 gradient of a widened bf16 input rounded to nearest even)"""
    return [g.to(dt) if g is not None and g.dtype != dt else g for g, dt in zip(grads, dtypes)]


def _ws(nbytes, dev):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)


def _flat_rows(x, name):
    x = _check(x, name)
    if x.dim() < 2:
        raise ValueError(f"{name}: expected [batch, ...], got shape {tuple(x.shape)}")
    return x.reshape(x.shape[0], -1)


def _same(a, b):
    return a is b or (a.data_ptr() == b.data_ptr() and a.shape == b.shape)


# ------------------------------------------------------------------------------------------------
# cost matrix: cost_xy / modified_cost / bi_causal_modified_cost
# ------------------------------------------------------------------------------------------------
class CostFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y, h1, M1, h2, M2, s):
        X, Y = _flat_rows(x, "x"), _flat_rows(y, "y")
        if X.shape[1] != Y.shape[1]:
            raise ValueError(f"x and y disagree on the feature size: {tuple(x.shape)} vs {tuple(y.shape)}")
        same = _same(X, Y)
        if same:
            Y = X
        Bx, K = X.shape
        By = Y.shape[0]
        pairs = []
        T = J = 0
        for h, M, tag in ((h1, M1, "1"), (h2, M2, "2")):
            if h is None:
                pairs.append((None, None))
                continue
            h, M = _check(h, "h" + tag, 3), _check(M, "M" + tag, 3)
            if h.shape[0] != Bx or M.shape[0] != By or h.shape[1:] != M.shape[1:]:
                raise ValueError(f"h{tag}/M{tag} shapes {tuple(h.shape)}/{tuple(M.shape)} do not match x/y batches "
                                 f"{Bx}/{By}")
            if T and (h.shape[1], h.shape[2]) != (T, J):
                raise ValueError("both martingale pairs must share [T, J]")
            T, J = h.shape[1], h.shape[2]
            pairs.append((h, M))
        dev = X.device
        C = torch.empty((Bx, By), dtype=torch.float32, device=dev)
        lib = _lib.load()
        nb = lib.kccot_cost_workspace_bytes(1, Bx, By, K)
        ws = _ws(nb, dev)
        with _on_device(dev):
            _lib.call("kccot_cost_fwd", _ptr(X), _ptr(Y), 1, Bx, By, K, _ptr(pairs[0][0]), _ptr(pairs[0][1]),
                      _ptr(pairs[1][0]), _ptr(pairs[1][1]), T, J, float(s), _ptr(C), _ptr(ws), ws.numel(),
                      _PATH["flags"], _stream(dev))
        ctx.save_for_backward(X, Y, *[t for p in pairs for t in p if t is not None])
        ctx.meta = (x.shape, y.shape, same, [p[0] is not None for p in pairs], T, J, float(s))
        return C

    @staticmethod
    def backward(ctx, gC):
        xshape, yshape, same, has, T, J, s = ctx.meta
        saved = list(ctx.saved_tensors)
        X, Y = saved[0], saved[1]
        rest = saved[2:]
        pairs = []
        for hflag in has:
            pairs.append((rest.pop(0), rest.pop(0)) if hflag else (None, None))
        gC = gC.contiguous().float()
        dev = X.device
        Bx, K = X.shape
        By = Y.shape[0]
        need = ctx.needs_input_grad
        gx = gy = None
        with _on_device(dev):
            st = _stream(dev)
            if need[0] or need[1]:
                gx = torch.empty_like(X) if need[0] else None
                gy = torch.empty_like(Y) if need[1] else None
                ws = _ws(_lib.load().kccot_cost_bwd_workspace_bytes(1, Bx, By, K), dev)
                _lib.call("kccot_cost_bwd", _ptr(gC), _ptr(X), _ptr(Y), 1, Bx, By, K, s, _ptr(gx), _ptr(gy),
                          _ptr(ws), ws.numel(), _PATH["flags"] if not same else _lib.PATH_SIMT, st)
            gout = [None, None, None, None]
            for q, (h, M) in enumerate(pairs):
                if h is None or not (need[2 + 2 * q] or need[3 + 2 * q]):
                    continue
                gh = torch.empty_like(h) if need[2 + 2 * q] else None
                gM = torch.empty_like(M) if need[3 + 2 * q] else None
                _lib.call("kccot_martingale_bwd", _ptr(gC), _ptr(h), _ptr(M), 1, Bx, By, T, J, s, _ptr(gh), _ptr(gM),
                          0, st)
                gout[2 * q], gout[2 * q + 1] = gh, gM
        gx = gx.reshape(xshape) if gx is not None else None
        gy = gy.reshape(yshape) if gy is not None else None
        return (gx, gy, *gout, None)


# ------------------------------------------------------------------------------------------------
# Sinkhorn solve on a given cost: C [n,B,B] -> cost [n]
# ------------------------------------------------------------------------------------------------
class SinkhornFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, C, eps, L, Lmin, thresh, exit_on_index):
        C = _check(C, "C", 3)
        n, B, B2 = C.shape
        if B != B2:
            raise ValueError(f"Sinkhorn needs square cost matrices, got {tuple(C.shape)}")
        dev = C.device
        L = int(L)
        uh = torch.empty((n, L + 1, B), dtype=torch.float32, device=dev)
        vh = torch.empty((n, L + 1, B), dtype=torch.float32, device=dev)
        nits = torch.empty((n,), dtype=torch.int32, device=dev)
        cost = torch.empty((n,), dtype=torch.float32, device=dev)
        ws = _ws(_lib.load().kccot_sinkhorn_workspace_bytes(n, B, L), dev)
        with _on_device(dev):
            _lib.call("kccot_sinkhorn_fwd", _ptr(C), n, B, float(eps), L, int(Lmin), float(thresh),
                      int(bool(exit_on_index)), _ptr(uh), _ptr(vh), _ptr(nits), _ptr(cost), _ptr(ws), ws.numel(),
                      _stream(dev))
        ctx.save_for_backward(C, uh, vh, nits)
        ctx.meta = (float(eps), L)
        ctx.mark_non_differentiable(nits)
        return cost, nits

    @staticmethod
    def backward(ctx, gcost, _gnits):
        C, uh, vh, nits = ctx.saved_tensors
        eps, L = ctx.meta
        n, B, _ = C.shape
        dev = C.device
        gcost = gcost.contiguous().float()
        Cbar = torch.empty_like(C)
        ws = _ws(_lib.load().kccot_sinkhorn_workspace_bytes(n, B, L), dev)
        with _on_device(dev):
            _lib.call("kccot_sinkhorn_bwd", _ptr(C), n, B, eps, L, _ptr(uh), _ptr(vh), _ptr(nits), _ptr(gcost),
                      _ptr(Cbar), _ptr(ws), ws.numel(), _stream(dev))
        return Cbar, None, None, None, None, None


# ------------------------------------------------------------------------------------------------
# fused mixed loss: 2*S(real,fake) - S(real,real) - S(fake,fake), one pass over the videos
# ------------------------------------------------------------------------------------------------
_SIZES = {}


def _mixed_sizes(B, K, L, nprob=1, dtype=torch.float32):
    """(saved, workspace) bytes; bf16 videos: the workspace depends on the path flag (native or widened path)"""
    bf16 = dtype == torch.bfloat16
    flags = _PATH["flags"] if bf16 else 0
    key = (B, K, L, nprob, dtype, flags)
    if key not in _SIZES:
        lib = _lib.load()
        ws = (lib.kccot_mixed_loss_workspace_bytes_bf16(nprob, B, K, L, flags) if bf16
              else lib.kccot_mixed_loss_workspace_bytes(nprob, B, K, L))
        _SIZES[key] = (int(lib.kccot_mixed_loss_saved_bytes(nprob, B, L)), int(ws))
    return _SIZES[key]


class MixedLossFn(torch.autograd.Function):
    """One C-ABI call per direction (kccot_mixed_loss_fwd_ctx / _bwd_ctx, or their _bf16 forms for bf16 videos)."""

    @staticmethod
    def forward(ctx, real, fake, h_fake, m_real, h_real, m_fake, s, eps, L, shared=(0, 0)):
        """shared = (period, len) in flattened columns: the shared-context hint of kccot_mixed_loss_*_ctx."""
        dtypes = [t.dtype if isinstance(t, torch.Tensor) else None for t in (real, fake, h_fake, m_real, h_real, m_fake)]
        R, F, bf16 = _videos(real, fake)
        if R.dim() < 2 or F.dim() < 2:
            raise ValueError(f"f_real / f_fake: expected [batch, ...], got shapes {tuple(real.shape)} / "
                             f"{tuple(fake.shape)}")
        R, F = R.reshape(R.shape[0], -1), F.reshape(F.shape[0], -1)
        if R.shape != F.shape:
            raise ValueError(f"f_real and f_fake must have the same shape, got {tuple(real.shape)} vs "
                             f"{tuple(fake.shape)}")
        B, K = R.shape
        hs = [_check_hm(t, n, 3) for t, n in ((h_fake, "h_fake"), (m_real, "m_real"), (h_real, "h_real"),
                                              (m_fake, "m_fake"))]
        T, J = hs[0].shape[1], hs[0].shape[2]
        for t, n in zip(hs, ("h_fake", "m_real", "h_real", "m_fake")):
            if tuple(t.shape) != (B, T, J):
                raise ValueError(f"{n}: expected shape {(B, T, J)}, got {tuple(t.shape)}")
        if T < 2:
            raise ValueError(f"the martingale term needs at least 2 time steps, got T={T}")
        dev = R.device
        L = int(L)
        saved_bytes, ws_bytes = _mixed_sizes(B, K, L, dtype=R.dtype)
        saved = torch.empty(saved_bytes, dtype=torch.uint8, device=dev)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        out = torch.empty(4, dtype=torch.float32, device=dev)          # loss | xy, xx, yy
        with _on_device(dev):
            _lib.call("kccot_mixed_loss_fwd_bf16" if bf16 else "kccot_mixed_loss_fwd_ctx", _ptr(R), _ptr(F), 1, B, K,
                      _ptr(hs[0]), _ptr(hs[1]), _ptr(hs[2]), _ptr(hs[3]), T, J, float(s), float(eps), L, _ptr(saved),
                      ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(out.data_ptr() + 4), _ptr(ws), ws_bytes,
                      _PATH["flags"], _stream(dev), int(shared[0]), int(shared[1]))
        ctx.save_for_backward(R, F, *hs, saved)
        ctx.meta = (real.shape, fake.shape, float(s), float(eps), L, (int(shared[0]), int(shared[1])), dtypes)
        loss, terms = out[0], out[1:]
        ctx.mark_non_differentiable(terms)
        ctx.set_materialize_grads(False)          # no zero-fill kernel for the unused gradient of `terms`
        return loss, terms

    @staticmethod
    def backward(ctx, gloss, _gterms):
        R, F, h_fake, m_real, h_real, m_fake, saved = ctx.saved_tensors
        rshape, fshape, s, eps, L, shared, dtypes = ctx.meta
        bf16 = R.dtype == torch.bfloat16
        B, K = R.shape
        T, J = h_fake.shape[1], h_fake.shape[2]
        dev = R.device
        need = ctx.needs_input_grad
        if gloss is None:                         # loss itself unused downstream
            return (None,) * 10
        gloss = gloss.reshape(1)
        if gloss.dtype != torch.float32 or not gloss.is_contiguous():
            gloss = gloss.float().contiguous()
        g_real = torch.empty_like(R) if need[0] else None
        g_fake = torch.empty_like(F) if need[1] else None
        gh_fake = torch.empty_like(h_fake) if need[2] else None
        gm_real = torch.empty_like(m_real) if need[3] else None
        gh_real = torch.empty_like(h_real) if need[4] else None
        gm_fake = torch.empty_like(m_fake) if need[5] else None
        _, ws_bytes = _mixed_sizes(B, K, L, dtype=R.dtype)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        with _on_device(dev):
            _lib.call("kccot_mixed_loss_bwd_bf16" if bf16 else "kccot_mixed_loss_bwd_ctx", _ptr(gloss), _ptr(R),
                      _ptr(F), 1, B, K, _ptr(h_fake), _ptr(m_real), _ptr(h_real), _ptr(m_fake), T, J, s, eps, L,
                      _ptr(saved), _ptr(g_real), _ptr(g_fake), _ptr(gh_fake), _ptr(gm_real), _ptr(gh_real),
                      _ptr(gm_fake), _ptr(ws), ws_bytes, _PATH["flags"], _stream(dev), shared[0], shared[1])
        g_real = g_real.reshape(rshape) if g_real is not None else None
        g_fake = g_fake.reshape(fshape) if g_fake is not None else None
        grads = _as_dtypes((g_real, g_fake, gh_fake, gm_real, gh_real, gm_fake), dtypes)
        return (*grads, None, None, None, None)


# ------------------------------------------------------------------------------------------------
# martingale penalty
# ------------------------------------------------------------------------------------------------
class MixedLossBatchedFn(torch.autograd.Function):
    """`nprob` independent problems in one C-ABI call per direction (BASELINE config 4): every tensor carries a
    leading problem axis, the result is one loss per problem."""

    @staticmethod
    def forward(ctx, real, fake, h_fake, m_real, h_real, m_fake, s, eps, L):
        dtypes = [t.dtype if isinstance(t, torch.Tensor) else None for t in (real, fake, h_fake, m_real, h_real, m_fake)]
        real, fake, bf16 = _videos(real, fake)
        if real.dim() < 3 or real.shape != fake.shape:
            raise ValueError(f"f_real / f_fake: expected equal shapes [nprob, B, ...], got {tuple(real.shape)} vs "
                             f"{tuple(fake.shape)}")
        P, B = real.shape[0], real.shape[1]
        R, F = real.reshape(P, B, -1), fake.reshape(P, B, -1)
        K = R.shape[2]
        hs = [_check_hm(t, n, 4) for t, n in ((h_fake, "h_fake"), (m_real, "m_real"), (h_real, "h_real"),
                                              (m_fake, "m_fake"))]
        T, J = hs[0].shape[2], hs[0].shape[3]
        for t, n in zip(hs, ("h_fake", "m_real", "h_real", "m_fake")):
            if tuple(t.shape) != (P, B, T, J):
                raise ValueError(f"{n}: expected shape {(P, B, T, J)}, got {tuple(t.shape)}")
        if T < 2:
            raise ValueError(f"the martingale term needs at least 2 time steps, got T={T}")
        dev = R.device
        L = int(L)
        saved_bytes, ws_bytes = _mixed_sizes(B, K, L, P, R.dtype)
        saved = torch.empty(saved_bytes, dtype=torch.uint8, device=dev)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        loss = torch.empty(P, dtype=torch.float32, device=dev)
        terms = torch.empty((P, 3), dtype=torch.float32, device=dev)
        with _on_device(dev):
            args = (_ptr(R), _ptr(F), P, B, K, _ptr(hs[0]), _ptr(hs[1]), _ptr(hs[2]), _ptr(hs[3]), T, J, float(s),
                    float(eps), L, _ptr(saved), _ptr(loss), _ptr(terms), _ptr(ws), ws_bytes, _PATH["flags"], _stream(dev))
            if bf16:
                _lib.call("kccot_mixed_loss_fwd_bf16", *args, 0, 0)
            else:
                _lib.call("kccot_mixed_loss_fwd", *args)
        ctx.save_for_backward(R, F, *hs, saved)
        ctx.meta = (real.shape, fake.shape, float(s), float(eps), L, dtypes)
        ctx.mark_non_differentiable(terms)
        ctx.set_materialize_grads(False)
        return loss, terms

    @staticmethod
    def backward(ctx, gloss, _gterms):
        R, F, h_fake, m_real, h_real, m_fake, saved = ctx.saved_tensors
        rshape, fshape, s, eps, L, dtypes = ctx.meta
        bf16 = R.dtype == torch.bfloat16
        P, B, K = R.shape
        T, J = h_fake.shape[2], h_fake.shape[3]
        dev = R.device
        need = ctx.needs_input_grad
        if gloss is None:
            return (None,) * 9
        gloss = gloss.reshape(P).float().contiguous()
        outs = [torch.empty_like(t) if need[i] else None for i, t in enumerate((R, F, h_fake, m_real, h_real, m_fake))]
        _, ws_bytes = _mixed_sizes(B, K, L, P, R.dtype)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        with _on_device(dev):
            args = (_ptr(gloss), _ptr(R), _ptr(F), P, B, K, _ptr(h_fake), _ptr(m_real), _ptr(h_real), _ptr(m_fake), T,
                    J, s, eps, L, _ptr(saved), *[_ptr(o) for o in outs], _ptr(ws), ws_bytes, _PATH["flags"], _stream(dev))
            if bf16:
                _lib.call("kccot_mixed_loss_bwd_bf16", *args, 0, 0)
            else:
                _lib.call("kccot_mixed_loss_bwd", *args)
        if outs[0] is not None:
            outs[0] = outs[0].reshape(rshape)
        if outs[1] is not None:
            outs[1] = outs[1].reshape(fshape)
        return (*_as_dtypes(outs, dtypes), None, None, None)


class MartingalePenaltyFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, M, reg_lam, s):
        M = _check(M, "M", 3)
        B, T, J = M.shape
        if T < 2:
            raise ValueError(f"M needs at least 2 time steps, got shape {tuple(M.shape)}")
        dev = M.device
        pm = torch.empty((), dtype=torch.float32, device=dev)
        stats = torch.empty((2 * J + (T - 1) * J,), dtype=torch.float32, device=dev)
        with _on_device(dev):
            _lib.call("kccot_pm_fwd", _ptr(M), B, T, J, float(reg_lam), float(s), _ptr(pm), _ptr(stats), _stream(dev))
        ctx.save_for_backward(M, stats)
        ctx.meta = (float(reg_lam), float(s))
        return pm

    @staticmethod
    def backward(ctx, gpm):
        M, stats = ctx.saved_tensors
        lam, s = ctx.meta
        B, T, J = M.shape
        gM = torch.empty_like(M)
        gpm = gpm.reshape(1).contiguous().float()
        with torch.cuda.device(M.device):
            _lib.call("kccot_pm_bwd", _ptr(M), B, T, J, lam, s, _ptr(stats), _ptr(gpm), _ptr(gM), _stream(M.device))
        return gM, None, None


class MartingalePenaltyBatchedFn(torch.autograd.Function):
    """`nprob` independent penalties in one C-ABI call per direction (kccot_pm_batched_fwd / _bwd): M is
    [nprob, B, T, J], the result [nprob], entry p the penalty of M[p] alone with the bits of a single call on it.  A bf16
    M is widened with .float() (exact) and its gradient comes back in bf16."""

    @staticmethod
    def forward(ctx, M, reg_lam, s):
        dtype = M.dtype if isinstance(M, torch.Tensor) else None
        M = _check_hm(M, "M", 4)
        P, B, T, J = M.shape
        if T < 2:
            raise ValueError(f"M needs at least 2 time steps, got shape {tuple(M.shape)}")
        dev = M.device
        pm = torch.empty((P,), dtype=torch.float32, device=dev)
        stats = torch.empty((P, 2 * J + (T - 1) * J), dtype=torch.float32, device=dev)
        with _on_device(dev):
            _lib.call("kccot_pm_batched_fwd", _ptr(M), P, B, T, J, float(reg_lam), float(s), _ptr(pm), _ptr(stats),
                      _stream(dev))
        ctx.save_for_backward(M, stats)
        ctx.meta = (float(reg_lam), float(s), dtype)
        return pm

    @staticmethod
    def backward(ctx, gpm):
        M, stats = ctx.saved_tensors
        lam, s, dtype = ctx.meta
        P, B, T, J = M.shape
        gM = torch.empty_like(M)
        gpm = gpm.reshape(P).float().contiguous()
        with _on_device(M.device):
            _lib.call("kccot_pm_batched_bwd", _ptr(M), P, B, T, J, lam, s, _ptr(stats), _ptr(gpm), _ptr(gM),
                      _stream(M.device))
        return gM.to(dtype), None, None


# ------------------------------------------------------------------------------------------------
# Gaussian smoothing
# ------------------------------------------------------------------------------------------------
def _taps(w):
    """Host weights -> (ctypes float array, radius); None -> (None, 0)."""
    if w is None:
        return None, 0
    arr = (ctypes.c_float * len(w))(*[float(v) for v in w])
    return arr, (len(w) - 1) // 2


class SmoothFn(torch.autograd.Function):
    """mode 1: `taps_t` filters T; mode 3: `taps_s` filters H, T and W.  The weights are host sequences (they become
    kernel arguments: nothing is copied to the device, so an annealed sigma costs nothing per step), or a
    data_utils.SmoothingTaps, whose device buffer the kernels read when they run (the *_dev entry points): a captured
    graph then follows its .set().  The forward snapshots that buffer (a device-to-device copy, capturable) and the
    backward filters with the snapshot, so a .set() between the two cannot change the gradient.
    A bf16 x runs kccot_smooth_fwd_bf16 / _bwd_bf16: output and gradient are bf16, and the tie mask of the forward (the
    elements at the maximum, which the bf16 output cannot tell apart from values just below it) is saved for the
    backward."""

    @staticmethod
    def _weights(ctx, taps_t, taps_s):
        """-> (entry-point suffix, weight arguments) for the taps saved on ctx"""
        if ctx.taps_dev is not None:
            return "_dev", (_ptr(ctx.taps_dev), ctx.radius)
        at, rt = _taps(taps_t)
        as_, rs = _taps(taps_s)
        return "", (at, rt, as_, rs)

    @staticmethod
    def forward(ctx, x, mode, taps_t, taps_s):
        x = _check_video(x, "inputs", 5)
        bf16 = x.dtype == torch.bfloat16
        B, H, T, W, C = x.shape
        dev = x.device
        lib = _lib.load()
        from .data_utils import SmoothingTaps
        taps = taps_t if mode == 1 else taps_s
        ctx.taps_dev = None
        if isinstance(taps, SmoothingTaps):
            if taps.weights.device != dev:
                raise ValueError(f"taps: the weights are on {taps.weights.device}, the video on {dev}")
            ctx.taps_dev, ctx.radius = taps.weights.clone(), taps.radius
        out = torch.empty_like(x)
        maxval = torch.empty((1,), dtype=torch.float32, device=dev)
        ws = _ws(lib.kccot_smooth_workspace_bytes(mode, B, H, T, W, C), dev)
        suffix, wargs = SmoothFn._weights(ctx, taps_t, taps_s)
        with _on_device(dev):
            if bf16:
                ties = torch.empty(lib.kccot_smooth_ties_bytes(B, H, T, W, C) // 4, dtype=torch.int32, device=dev)
                _lib.call("kccot_smooth_fwd_bf16" + suffix, mode, _ptr(x), B, H, T, W, C, *wargs, _ptr(out),
                          _ptr(maxval), _ptr(ties), _ptr(ws), ws.numel(), _stream(dev))
                ctx.save_for_backward(out, maxval, ties)
            else:
                _lib.call("kccot_smooth_fwd" + suffix, mode, _ptr(x), B, H, T, W, C, *wargs, _ptr(out), _ptr(maxval),
                          _ptr(ws), ws.numel(), _stream(dev))
                ctx.save_for_backward(out, maxval)
        ctx.mode, ctx.taps = mode, (taps_t, taps_s)
        return out

    @staticmethod
    def backward(ctx, gout):
        out, maxval, *ties = ctx.saved_tensors
        B, H, T, W, C = out.shape
        dev = out.device
        gout = gout.contiguous().to(out.dtype)
        gx = torch.empty_like(out)
        ws = _ws(_lib.load().kccot_smooth_workspace_bytes(ctx.mode, B, H, T, W, C), dev)
        suffix, wargs = SmoothFn._weights(ctx, *ctx.taps)
        with _on_device(dev):
            if ties:
                _lib.call("kccot_smooth_bwd_bf16" + suffix, ctx.mode, _ptr(gout), _ptr(out), _ptr(maxval),
                          _ptr(ties[0]), B, H, T, W, C, *wargs, _ptr(gx), _ptr(ws), ws.numel(), _stream(dev))
            else:
                _lib.call("kccot_smooth_bwd" + suffix, ctx.mode, _ptr(gout), _ptr(out), _ptr(maxval), B, H, T, W, C,
                          *wargs, _ptr(gx), _ptr(ws), ws.numel(), _stream(dev))
        return gx, None, None, None


class SmoothBatchedFn(torch.autograd.Function):
    """`nprob` independent smoothings in one call per direction (kccot_smooth_batched_fwd / _bwd): x is
    [nprob, B, H, T, W, C], `taps` a data_utils.SmoothingTaps with nprob rows, row p the weights of problem p, which is
    divided by its own maximum.  As in SmoothFn, mode 1 filters T and mode 3 filters H, T and W, the forward snapshots
    the weights for the backward, and a bf16 x runs the _bf16 entries and saves the tie mask of the whole batch."""

    @staticmethod
    def forward(ctx, x, mode, taps):
        x = _check_video(x, "inputs", 6)
        bf16 = x.dtype == torch.bfloat16
        P, B, H, T, W, C = x.shape
        dev = x.device
        if taps.weights.device != dev:
            raise ValueError(f"taps: the weights are on {taps.weights.device}, the video on {dev}")
        if tuple(taps.weights.shape) != (P, 2 * taps.radius + 1):
            raise ValueError(f"taps: weights of shape {tuple(taps.weights.shape)} for {P} problems of radius "
                             f"{taps.radius}; expected {(P, 2 * taps.radius + 1)}")
        lib = _lib.load()
        w = taps.weights.clone()
        out = torch.empty_like(x)
        maxval = torch.empty((P,), dtype=torch.float32, device=dev)
        ws = _ws(lib.kccot_smooth_batched_workspace_bytes(mode, P, B, H, T, W, C), dev)
        with _on_device(dev):
            if bf16:
                ties = torch.empty(lib.kccot_smooth_ties_bytes(P * B, H, T, W, C) // 4, dtype=torch.int32, device=dev)
                _lib.call("kccot_smooth_batched_fwd_bf16", mode, _ptr(x), P, B, H, T, W, C, _ptr(w), taps.radius,
                          _ptr(out), _ptr(maxval), _ptr(ties), _ptr(ws), ws.numel(), _stream(dev))
                ctx.save_for_backward(out, maxval, w, ties)
            else:
                _lib.call("kccot_smooth_batched_fwd", mode, _ptr(x), P, B, H, T, W, C, _ptr(w), taps.radius, _ptr(out),
                          _ptr(maxval), _ptr(ws), ws.numel(), _stream(dev))
                ctx.save_for_backward(out, maxval, w)
        ctx.mode, ctx.radius = mode, taps.radius
        return out

    @staticmethod
    def backward(ctx, gout):
        out, maxval, w, *ties = ctx.saved_tensors
        P, B, H, T, W, C = out.shape
        dev = out.device
        gout = gout.contiguous().to(out.dtype)
        gx = torch.empty_like(out)
        ws = _ws(_lib.load().kccot_smooth_batched_workspace_bytes(ctx.mode, P, B, H, T, W, C), dev)
        with _on_device(dev):
            if ties:
                _lib.call("kccot_smooth_batched_bwd_bf16", ctx.mode, _ptr(gout), _ptr(out), _ptr(maxval),
                          _ptr(ties[0]), P, B, H, T, W, C, _ptr(w), ctx.radius, _ptr(gx), _ptr(ws), ws.numel(),
                          _stream(dev))
            else:
                _lib.call("kccot_smooth_batched_bwd", ctx.mode, _ptr(gout), _ptr(out), _ptr(maxval), P, B, H, T, W, C,
                          _ptr(w), ctx.radius, _ptr(gx), _ptr(ws), ws.numel(), _stream(dev))
        return gx, None, None
