"""bf16 videos in the Gaussian kernel smoothing.  Needs a B200: `pytest -m gpu`.

Contract (include/kccot.h, kccot_smooth_*_bf16), for a bf16 input x:
  * forward, exact: out is the fp32 smoothing of x.float() rounded to nearest even (torch.equal), and maxval is
    bit-identical to the fp32 call's;
  * tie set, exact: the forward's bit mask marks the elements whose fp32 quotient is exactly 1.0, the set the fp32
    backward finds with out == 1.0.  The bf16 output cannot carry it (every fp32 value in [1 - 2^-9, 1) rounds to 1.0);
  * backward: gx (bf16) equals the fp32 backward on gout.float(), rounded to nearest even, at every element outside
    the adjoint stencil's support of the tied maxima.  Inside it gx may differ only through S = sum(gout * out), which
    the bf16 path forms from the bf16 out; everywhere gx is held to the fp64 oracle within GRAD_TOL_BF16, a few
    units of bf16 rounding (2^-9 relative per element) in rel-L2.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_l2

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
GRAD_TOL_BF16 = 4e-3


@pytest.fixture(scope="module", autouse=True)
def _device():
    from kccotgan_b200 import _lib
    assert _lib.load().kccot_device_check() == 0, _lib.last_error()


def _ks(tk=6, sk=6):
    from kccotgan_b200.data_utils import KernelSmoothing
    return KernelSmoothing(temporal_kernel_size=tk, spatial_kernel_size=sk)


def _fns(ks):
    from oracle import closed_form as cf
    return (("1d", ks.temporal_convolution, cf.temporal_convolution, ks.temporal_radius),
            ("3d", ks.gaussian_convolution3D, cf.gaussian_convolution3D, ks.spatial_radius))


def _fwd_bwd(fn, x, gout, sigma):
    xl = x.detach().requires_grad_(True)                       # same storage and offset as x
    out = fn(xl, sigma)
    gx, = torch.autograd.grad(out, xl, gout)
    torch.cuda.synchronize()
    return out.detach(), gx


def _support(tie, mode, radius, sigma):
    """elements of gx that the tied maxima reach through the adjoint passes (nonzero pattern of A^T per axis)"""
    from oracle import closed_form as cf
    z = tie.astype(np.float64)
    axes = (2,) if mode == "1d" else (1, 2, 3)
    for axis in axes:
        nz = (cf._filter_matrix(z.shape[axis], radius, sigma) != 0).astype(np.float64)
        z = cf._apply_axis(z, nz.T, axis)
    return z > 0


def _check_exact(mode, r, sigma, shape, out16, gx16, out32, gx32):
    assert out16.dtype == BF and gx16.dtype == BF
    assert torch.equal(out16, out32.to(BF)), (mode, shape)
    outside = torch.from_numpy(~_support((out32 == 1.0).cpu().numpy(), mode, r, sigma)).cuda()
    want = gx32.to(BF)
    if not torch.equal(gx16[outside], want[outside]):
        diff = (gx16[outside].view(torch.int16).int() - want[outside].view(torch.int16).int()).abs()
        pytest.fail(f"{mode} {shape}: {int((diff != 0).sum())} elements outside the tie support differ, "
                    f"max {int(diff.max())} bf16 ulps")


def _assert_contract(ks, x, gout, sigma, oracle=True):
    """x, gout: bf16 CUDA tensors.  Checks forward exactness, backward exactness outside the tie support and the fp64
    oracle, for both modes."""
    for mode, fn, cfn, r in _fns(ks):
        out16, gx16 = _fwd_bwd(fn, x, gout, sigma)
        out32, gx32 = _fwd_bwd(fn, x.float(), gout.float(), sigma)
        _check_exact(mode, r, sigma, tuple(x.shape), out16, gx16, out32, gx32)
        if oracle:
            xo, go = (t.float().cpu().numpy().astype(np.float64) for t in (x, gout))
            _, rg = cfn(xo, sigma, radius=r, grad_out=go)
            e = rel_l2(gx16.float().cpu().numpy(), rg)
            assert e < GRAD_TOL_BF16, (mode, tuple(x.shape), e)


def _draw(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(shape, generator=g).to(BF).cuda(), torch.randn(shape, generator=g).to(BF).cuda()


# ---------------------------------------------------------------------------------------------
# forward exactness and backward, across the kernels' shapes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(2, 9, 7, 10, 1), (3, 16, 5, 12, 3), (1, 4, 4, 5, 2), (2, 64, 20, 64, 1),
                                   (2, 12, 9, 7, 4), (5, 8, 64, 6, 1)])
def test_shapes(shape):
    """the shapes of the fp32 smoothing tests: both filter kernels, the 16-byte and scalar paths, single channels"""
    _assert_contract(_ks(), *_draw(shape, sum(shape)), 2.5)


@pytest.mark.parametrize("tk,sk,shape", [
    (8, 8, (2, 12, 10, 12, 3)),
    (6, 8, (2, 16, 7, 16, 1)),
    (2, 3, (3, 6, 5, 6, 2)),          # radius 1
    (12, 12, (1, 16, 14, 16, 1)),     # radius 6
    (6, 6, (1, 96, 8, 80, 1)),        # axes longer than 64
    (6, 6, (1, 8, 200, 4, 1)),        # a long temporal axis
    (4, 10, (2, 14, 9, 11, 3)),       # radii 2 and 5, inner % 4 != 0
])
def test_radius_and_axis_range(tk, sk, shape):
    _assert_contract(_ks(tk, sk), *_draw(shape, tk * 100 + sk), 2.0)


def test_config3_full_tensor():
    """[64, 64, 12, 64, 3], the BAIR shape of config 3; the oracle on a quarter of the batch (fp64 on the CPU)"""
    x, go = _draw((64, 64, 12, 64, 3), 3)
    _assert_contract(_ks(), x, go, 5.0, oracle=False)
    _assert_contract(_ks(), x[:16].contiguous(), go[:16].contiguous(), 5.0)


def test_misaligned_view():
    """a view with a storage offset of one element (2 bytes): the kernels take their scalar paths"""
    shape = (2, 16, 8, 16, 3)
    n = int(np.prod(shape))
    x, go = _draw((n + 1,), 11)
    xv, gv = x[1:].view(shape), go[1:].view(shape)
    assert xv.data_ptr() % 16 == 2
    _assert_contract(_ks(), xv, gv, 3.0)


# ---------------------------------------------------------------------------------------------
# the tie set
# ---------------------------------------------------------------------------------------------
def _abi(mode, x, ks, sigma):
    """kccot_smooth_fwd_bf16 and kccot_smooth_fwd (on x.float()) called directly -> (out16, max16, ties, out32, max32)"""
    from kccotgan_b200 import _lib
    from kccotgan_b200.functional import _ptr, _stream, _taps
    lib = _lib.load()
    B, H, T, W, C = x.shape
    taps = tuple(ks._weights(ks.temporal_radius if mode == 1 else ks.spatial_radius, sigma))
    (at, rt), (as_, rs) = (_taps(taps), _taps(None)) if mode == 1 else (_taps(None), _taps(taps))
    ws = torch.empty(max(256, lib.kccot_smooth_workspace_bytes(mode, B, H, T, W, C)), dtype=torch.uint8, device="cuda")
    out16, out32 = torch.empty_like(x), torch.empty(x.shape, device="cuda")
    max16, max32 = torch.empty(1, device="cuda"), torch.empty(1, device="cuda")
    ties = torch.full((lib.kccot_smooth_ties_bytes(B, H, T, W, C) // 4,), -1, dtype=torch.int32, device="cuda")
    st = _stream(x.device)
    _lib.call("kccot_smooth_fwd_bf16", mode, _ptr(x), B, H, T, W, C, at, rt, as_, rs, _ptr(out16), _ptr(max16),
              _ptr(ties), _ptr(ws), ws.numel(), st)
    xf = x.float()
    _lib.call("kccot_smooth_fwd", mode, _ptr(xf), B, H, T, W, C, at, rt, as_, rs, _ptr(out32), _ptr(max32), _ptr(ws),
              ws.numel(), st)
    torch.cuda.synchronize()
    return out16, max16, ties, out32, max32


def _unpack(ties, n):
    w = ties.cpu().numpy().view(np.uint32)
    return np.unpackbits(w.view(np.uint8), bitorder="little")[:n].astype(bool)


@pytest.mark.parametrize("mode", [1, 3])
@pytest.mark.parametrize("shape", [(2, 9, 7, 10, 1), (2, 64, 12, 64, 3), (1, 8, 200, 4, 1)])
def test_maxval_and_tie_mask(mode, shape):
    """maxval bit-identical; the mask (zeroed by the call: it starts all ones here) is exactly out32 == 1.0"""
    x, _ = _draw(shape, 5)
    ks = _ks()
    out16, max16, ties, out32, max32 = _abi(mode, x, ks, 2.5)
    assert torch.equal(max16, max32)
    assert torch.equal(out16, out32.to(BF))
    n = x.numel()
    assert np.array_equal(_unpack(ties, n), (out32 == 1.0).cpu().numpy().reshape(-1))
    assert not _unpack(ties, ties.numel() * 32)[n:].any()


@pytest.mark.parametrize("sigma", [5.0, 1.7])
def test_golden_tie_case(sigma):
    """x_tie of the golden file has several exact maxima: the popcount of the mask is the fp32 tie count, and the
    gradient meets the oracle"""
    g = load_golden("smoothing.npz")
    x = torch.from_numpy(g["x_tie"]).to(BF).cuda()
    go = torch.from_numpy(g["gout_tie"]).to(BF).cuda()
    ks = _ks()
    for mode in (1, 3):
        out16, _, ties, out32, _ = _abi(mode, x, ks, sigma)
        count = int((out32 == 1.0).sum())
        assert count >= 2, (mode, count)
        assert int(_unpack(ties, x.numel()).sum()) == count
    _assert_contract(ks, x, go, sigma)


@pytest.mark.parametrize("W", [2, 64])
def test_near_tie_gets_no_tie_term(W):
    """Element b's smoothed value is 1 - 2^-10 of the maximum at element a: not a tie, but it rounds to 1.0 in bf16.
    The gradient at b's column must be the fp32 one, i.e. no tie term there (a design that took the ties from the
    bf16 output would split the max gradient between a and b).  W = 2 runs the tile kernel, W = 64 the column kernel."""
    ks = _ks()
    sigma = 5.0
    w = ks._weights(ks.temporal_radius, sigma).astype(np.float64)
    x = torch.zeros(1, 2, 12, W, 1)                           # t = 6: out of reach of the REFLECT padding
    x[0, 0, 6, 0, 0] = 1.0                                    # a: the maximum, exactly w[3]
    x[0, 0, 6, 1, 0] = 1.0 - 2.0 ** -8                        # b: 1 - 2^-8 of it ...
    a = 0.375 * w[3] / w[2] * 2.0 ** -8                       # ... plus 3/4 of the gap from its two neighbours
    x[0, 0, 5, 1, 0] = a
    x[0, 0, 7, 1, 0] = a
    x = x.to(BF).cuda()
    out32 = ks.temporal_convolution(x.float(), sigma)
    vals = out32.flatten().sort(descending=True).values
    assert float(vals[0]) == 1.0 and 1.0 - 2.0 ** -9 <= float(vals[1]) < 1.0, vals[:2]
    assert int((out32.to(BF) == 1.0).sum()) == 2                # the bf16 output cannot tell b from a
    go = torch.randn(x.shape, generator=torch.Generator().manual_seed(9)).to(BF).cuda()
    out16, gx16 = _fwd_bwd(ks.temporal_convolution, x, go, sigma)
    _, gx32 = _fwd_bwd(ks.temporal_convolution, x.float(), go.float(), sigma)
    assert torch.equal(out16, out32.to(BF))
    assert torch.equal(gx16[..., 1:, :], gx32.to(BF)[..., 1:, :])    # b's column: outside the support of the tie
    _check_exact("1d", ks.temporal_radius, sigma, tuple(x.shape), out16, gx16, out32, gx32)
    from oracle import closed_form as cf                  # (1d only: H = 2 is too short for the 3-D filter)
    _, rg = cf.temporal_convolution(x.float().cpu().numpy().astype(np.float64), sigma,
                                    grad_out=go.float().cpu().numpy().astype(np.float64))
    assert rel_l2(gx16.float().cpu().numpy(), rg) < GRAD_TOL_BF16


# ---------------------------------------------------------------------------------------------
# graph capture, the config-3 chain, dtypes
# ---------------------------------------------------------------------------------------------
def test_graph_capture_with_annealed_sigma():
    """the taps are kernel arguments and the mask / sums are cleared with cudaMemsetAsync: forward and backward with
    a never-seen sigma replay from a CUDA graph"""
    ks = _ks()
    x, go = _draw((2, 8, 6, 8, 3), 21)
    sig = ks.annealing_sigma(5.0, 12345)
    for mode, fn, _, r in _fns(ks):
        _fwd_bwd(fn, x, go, 4.0)                                 # warm-up with a different sigma
        xl = x.detach().requires_grad_(True)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            out = fn(xl, sig)
            gx, = torch.autograd.grad(out, xl, go)
        gr.replay()
        torch.cuda.synchronize()
        out32, gx32 = _fwd_bwd(fn, x.float(), go.float(), sig)
        _check_exact(mode, r, sig, tuple(x.shape), out, gx, out32, gx32)


def test_config3_chain_in_bf16():
    """kernel_train.py's `--kernel 1d` step in bf16: smoothing of real and fake, the mixed loss, both adjoints.  The
    loss equals the fp32 loss on the smoothed bf16 videos widened (the mixed loss contract), and the video gradients
    are bf16 and meet the fp64 oracle of the whole chain."""
    from kccotgan_b200 import gan_utils
    from kccotgan_b200.synthetic import CONFIGS, make_inputs
    from oracle import closed_form as cf
    c = {k: v for k, v in CONFIGS["cfg3_bair"].items() if k not in ("nprob", "ctx")}
    inp = make_inputs(J=8, kind="uniform", seed=4, device="cuda", **c)
    ks = _ks()
    sigma, s = 5.0, 1.0 / 15.0
    real = inp["real"].to(BF).requires_grad_(True)
    fake = inp["fake"].to(BF).requires_grad_(True)
    hm = [inp[k] for k in ("h_fake", "m_real", "h_real", "m_fake")]
    rs, fs = ks.temporal_convolution(real, sigma), ks.temporal_convolution(fake, sigma)
    assert rs.dtype == fs.dtype == BF
    loss = gan_utils.compute_sinkhorn_loss(rs, fs, s, 0.8, 100, *hm)
    g_real, g_fake = torch.autograd.grad(loss, (real, fake))
    loss32 = gan_utils.compute_sinkhorn_loss(rs.detach().float(), fs.detach().float(), s, 0.8, 100, *hm)
    assert torch.equal(loss.detach(), loss32)
    assert g_real.dtype == g_fake.dtype == BF
    a = [t.detach().float().cpu().numpy().astype(np.float64) for t in (real, fake, *hm)]
    ro, fo = cf.temporal_convolution(a[0], sigma), cf.temporal_convolution(a[1], sigma)
    _, gref, _ = cf.compute_sinkhorn_loss(ro, fo, s, 0.8, 100, *a[2:], grad=True)
    _, gr = cf.temporal_convolution(a[0], sigma, grad_out=gref["f_real"])
    _, gf = cf.temporal_convolution(a[1], sigma, grad_out=gref["f_fake"])
    for name, got, ref in (("f_real", g_real, gr), ("f_fake", g_fake, gf)):
        e = rel_l2(got.float().cpu().numpy(), ref)
        assert e < 1e-2, (name, e)


@pytest.mark.parametrize("dtype", [torch.float16, torch.float64])
def test_other_dtypes_raise(dtype):
    ks = _ks()
    x = torch.rand(2, 8, 6, 8, 1, device="cuda").to(dtype)
    for fn in (ks.temporal_convolution, ks.gaussian_convolution3D):
        with pytest.raises(ValueError):
            fn(x, 2.0)


def test_bf16_cpu_tensor_raises():
    with pytest.raises(ValueError, match="CUDA"):
        _ks().temporal_convolution(torch.rand(2, 8, 6, 8, 1).to(BF), 2.0)
