"""Gaussian smoothing of batched independent problems (KernelSmoothing.*_batched, kccot_smooth_batched_*).  Needs a
B200: `pytest -m gpu`.

Contract: for each problem p of a [nprob, B, H, T, W, C] call, against the *_dev entry called on x[p] with weights
row p, out[p], maxval[p] and (bf16) the tie-mask bits of problem p are bit-identical; gx[p] is bit-identical outside the
adjoint stencil of p's tied maxima (inside it both sides sum S_p = sum(gout * out) with atomics in a run-dependent
order, held to the tolerance of test_gpu_smoothing_device_taps._assert_grad).  A tie in one problem changes no other
problem's numbers.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden
from test_gpu_bf16_smoothing import _unpack
from test_gpu_smoothing_device_taps import SHAPES, _abi, _assert_eager_equal, _assert_grad

pytestmark = pytest.mark.gpu

BF = torch.bfloat16


@pytest.fixture(scope="module", autouse=True)
def _device():
    from kccotgan_b200 import _lib
    assert _lib.load().kccot_device_check() == 0, _lib.last_error()


def _ks(r=3):
    from kccotgan_b200.data_utils import KernelSmoothing
    return KernelSmoothing(temporal_kernel_size=2 * r, spatial_kernel_size=2 * r)


def _sigmas(nprob, r):
    return [0.5 + r + 0.7 * p for p in range(nprob)]


def _batched_abi(mode, x, gout, r, sigmas):
    """forward and backward of kccot_smooth_batched_* -> (out, maxval [nprob], tie mask or None, gx)"""
    from kccotgan_b200 import _lib
    from kccotgan_b200.data_utils import SmoothingTaps
    from kccotgan_b200.functional import _ptr, _stream
    lib = _lib.load()
    P, B, H, T, W, C = x.shape
    w = SmoothingTaps(r, nprob=P).set(sigmas).weights
    ws = torch.empty(max(256, lib.kccot_smooth_batched_workspace_bytes(mode, P, B, H, T, W, C)), dtype=torch.uint8,
                     device="cuda")
    out, gx, mx = torch.empty_like(x), torch.empty_like(x), torch.empty(P, device="cuda")
    st = _stream(x.device)
    dims = (P, B, H, T, W, C)
    if x.dtype == BF:
        ties = torch.full((lib.kccot_smooth_ties_bytes(P * B, H, T, W, C) // 4,), -1, dtype=torch.int32, device="cuda")
        _lib.call("kccot_smooth_batched_fwd_bf16", mode, _ptr(x), *dims, _ptr(w), r, _ptr(out), _ptr(mx), _ptr(ties),
                  _ptr(ws), ws.numel(), st)
        _lib.call("kccot_smooth_batched_bwd_bf16", mode, _ptr(gout), _ptr(out), _ptr(mx), _ptr(ties), *dims, _ptr(w), r,
                  _ptr(gx), _ptr(ws), ws.numel(), st)
    else:
        ties = None
        _lib.call("kccot_smooth_batched_fwd", mode, _ptr(x), *dims, _ptr(w), r, _ptr(out), _ptr(mx), _ptr(ws),
                  ws.numel(), st)
        _lib.call("kccot_smooth_batched_bwd", mode, _ptr(gout), _ptr(out), _ptr(mx), *dims, _ptr(w), r, _ptr(gx),
                  _ptr(ws), ws.numel(), st)
    torch.cuda.synchronize()
    return out, mx, ties, gx


def _gout_like(x, seed):
    gout = torch.randn(x.shape, generator=torch.Generator().manual_seed(seed)).to(x.dtype).cuda()
    if x.data_ptr() % 16:                                   # keep gout's misalignment like x's
        g = torch.empty(x.numel() + 1, dtype=x.dtype, device="cuda")
        gout = g[1:].view(x.shape).copy_(gout)
    return gout


def _check_contract(mode, x, r, sigmas, seed=0, exact=()):
    """every problem against its single *_dev call; problems in `exact` bit for bit in gx as well
    -> the number of tied maxima of each problem"""
    P = x.shape[0]
    n = x[0].numel()
    gout = _gout_like(x, seed)
    out, mx, ties, gx = _batched_abi(mode, x, gout, r, sigmas)
    bits = _unpack(ties, P * n) if ties is not None else None
    if ties is not None:
        assert not _unpack(ties, ties.numel() * 32)[P * n:].any()
    counts = []
    for p in range(P):
        o1, m1, t1, g1 = _abi(mode, x[p], gout[p], r, sigmas[p], dev=True)
        assert torch.equal(out[p], o1), (mode, r, p, tuple(x.shape))
        assert torch.equal(mx[p:p + 1], m1), (mode, r, p)
        if t1 is not None:
            tie = _unpack(t1, n)
            assert np.array_equal(bits[p * n:(p + 1) * n], tie), (mode, r, p)
        else:
            tie = (o1 == 1.0).cpu().numpy().reshape(-1)
        assert tie.any()
        counts.append(int(tie.sum()))
        if p in exact:
            assert torch.equal(gx[p], g1), (mode, r, p)
        else:
            _assert_grad(mode, r, sigmas[p], tie, gx[p], g1)
    return counts


def _draw(shape, dtype, seed):
    return torch.rand(shape, generator=torch.Generator().manual_seed(seed)).to(dtype).cuda()


# the shapes of the device-weight tests (tile kernel, column kernels of 8 / 4 / 1 elements per thread), and one whose
# problem size is not a multiple of 32, so that tie-mask words straddle two problems
CASES = [(s, P) for s in SHAPES + [(2, 9, 7, 10, 1)] for P in (1, 3, 5) if not (s == SHAPES[3] and P == 5)]


@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
@pytest.mark.parametrize("r", [1, 3, 6])
@pytest.mark.parametrize("mode", [1, 3])
@pytest.mark.parametrize("shape,nprob", CASES)
def test_same_numbers_as_single_calls(shape, nprob, mode, r, dtype):
    x = _draw((nprob, *shape), dtype, sum(shape) + r + nprob)
    _check_contract(mode, x, r, _sigmas(nprob, r))


@pytest.mark.parametrize("mode", [1, 3])
def test_misaligned_bf16_view(mode):
    """a storage offset of one element (2 bytes): the bf16 kernels take their one-element paths"""
    shape = (3, 2, 16, 8, 16, 3)
    x = _draw((int(np.prod(shape)) + 1,), BF, 11)
    xv = x[1:].view(shape)
    assert xv.data_ptr() % 16 == 2
    _check_contract(mode, xv, 3, [3.0, 1.5, 4.0])


@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
@pytest.mark.parametrize("sigma", [5.0, 1.7])
def test_tie_in_one_problem_stays_there(dtype, sigma):
    """the golden tie case (several exact maxima) as problem 1 of 3: it meets the contract, and problems 0 and 2 come
    out bit-identical to their single calls in both directions (at this size both sides form each S_p in one CTA)"""
    g = load_golden("smoothing.npz")
    tie = torch.from_numpy(g["x_tie"])
    x = torch.stack([torch.rand(tie.shape, generator=torch.Generator().manual_seed(5)), tie,
                     torch.rand(tie.shape, generator=torch.Generator().manual_seed(6))]).to(dtype).cuda()
    for mode in (1, 3):
        ties = _check_contract(mode, x, 3, [sigma, sigma, 2.0], seed=4, exact=(0, 2))
        assert ties[1] >= 2, (mode, ties)


def _fwd_bwd(fn, x, gout, sigma):
    xl = x.detach().requires_grad_(True)
    out = fn(xl, sigma)
    gx, = torch.autograd.grad(out, xl, gout)
    return out.detach(), gx


@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
@pytest.mark.parametrize("mode", [1, 3])
def test_config4_full_size(mode, dtype):
    """256 x [64, 32, 10, 32, 1]: the forward against 256 single calls bit for bit, then smoothing ->
    compute_sinkhorn_loss_batched -> backward: the losses equal those of the stacked single outputs, and the gradient
    with respect to the raw fake videos meets the contract"""
    from kccotgan_b200 import gan_utils
    from kccotgan_b200.synthetic import CONFIGS
    c = CONFIGS["cfg4_batched"]
    P, B, H, T, W, C = c["nprob"], c["B"], c["H"], c["T"], c["W"], c["C"]
    ks = _ks()
    batched = ks.temporal_convolution_batched if mode == 1 else ks.gaussian_convolution3D_batched
    single = ks.temporal_convolution if mode == 1 else ks.gaussian_convolution3D
    r = ks.temporal_radius if mode == 1 else ks.spatial_radius
    sigmas = [ks.annealing_sigma(5.0, 40 * p) for p in range(P)]
    gen = torch.Generator(device="cuda").manual_seed(40)
    real = torch.rand((P, B, H, T, W, C), generator=gen, device="cuda").to(dtype)
    fake = torch.rand((P, B, H, T, W, C), generator=gen, device="cuda").to(dtype).requires_grad_(True)
    hm = [torch.sigmoid(torch.randn((P, B, T, 8), generator=gen, device="cuda")) for _ in range(4)]

    rs = batched(real, sigmas)
    fs = batched(fake, sigmas)
    rs1 = torch.stack([single(real[p], sigmas[p]) for p in range(P)])
    with torch.no_grad():
        fs1 = torch.stack([single(fake[p], sigmas[p]) for p in range(P)])
    assert torch.equal(rs, rs1) and torch.equal(fs.detach(), fs1)

    loss = gan_utils.compute_sinkhorn_loss_batched(rs, fs, 1.0 / 15.0, *hm)
    loss1 = gan_utils.compute_sinkhorn_loss_batched(rs1, fs1, 1.0 / 15.0, *hm)
    assert torch.equal(loss.detach(), loss1)
    gfs, gfake = torch.autograd.grad(loss.sum(), [fs, fake])
    assert gfake.dtype == dtype
    for p in range(P):                      # the single smoothing backward fed with the same upstream gradient
        o1, g1 = _fwd_bwd(single, fake[p].detach(), gfs[p], sigmas[p])
        _assert_eager_equal(mode, r, sigmas[p], fs[p].detach(), gfake[p], o1, g1)


@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
def test_graph_follows_set(dtype):
    """forward + backward of both batched smoothings captured once with a SmoothingTaps(r, nprob=3); every replay after
    a .set() of a different annealed sigma per problem equals the eager call at those sigmas"""
    from kccotgan_b200.data_utils import SmoothingTaps
    ks = _ks()
    P = 3
    x = _draw((P, 2, 16, 8, 16, 3), dtype, 21)
    gout = torch.randn(x.shape, generator=torch.Generator().manual_seed(22)).to(dtype).cuda()
    taps = SmoothingTaps(3, nprob=P).set(5.0)
    fns = ((1, ks.temporal_convolution_batched), (3, ks.gaussian_convolution3D_batched))
    xl = x.detach().requires_grad_(True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                               # warm-up outside the capture
        for _, fn in fns:
            torch.autograd.grad(fn(xl, taps), xl, gout)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        res = []
        for _, fn in fns:
            out = fn(xl, taps)
            gx, = torch.autograd.grad(out, xl, gout)
            res.append((out.detach(), gx))
    graph.replay()
    torch.cuda.synchronize()
    at_capture = [o.clone() for o, _ in res]
    for step in (0, 1, 500, 5000, 12345):
        sig = [ks.annealing_sigma(5.0, step + 700 * p) for p in range(P)]
        taps.set(sig)
        graph.replay()
        torch.cuda.synchronize()
        for (mode, fn), (out, gx), out0 in zip(fns, res, at_capture):
            out_ref, gx_ref = _fwd_bwd(fn, x, gout, sig)
            torch.cuda.synchronize()
            for p in range(P):
                _assert_eager_equal(mode, 3, sig[p], out[p], gx[p], out_ref[p], gx_ref[p])
            if step == 12345:
                assert not torch.equal(out, out0), mode          # the replay really filtered with other weights


@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
def test_sigma_forms_agree(dtype):
    """a number, a sequence of equal numbers and a SmoothingTaps set to that number give the same results"""
    from kccotgan_b200.data_utils import SmoothingTaps
    ks = _ks()
    x = _draw((4, 2, 16, 8, 16, 3), dtype, 31)
    gout = torch.randn(x.shape, generator=torch.Generator().manual_seed(32)).to(dtype).cuda()
    for mode, fn in ((1, ks.temporal_convolution_batched), (3, ks.gaussian_convolution3D_batched)):
        ref = _fwd_bwd(fn, x, gout, 2.5)
        assert ref[0].dtype == dtype and ref[1].dtype == dtype
        for sigma in ([2.5] * 4, (2.5,) * 4, np.float32(2.5), SmoothingTaps(3, nprob=4).set(2.5)):
            out, gx = _fwd_bwd(fn, x, gout, sigma)
            for p in range(4):
                _assert_eager_equal(mode, 3, 2.5, out[p], gx[p], ref[0][p], ref[1][p])


def test_bad_inputs_raise_without_a_launch():
    from kccotgan_b200 import _lib
    from kccotgan_b200.data_utils import SmoothingTaps
    lib = _lib.load()
    ks = _ks()
    x = _draw((3, 2, 16, 8, 16, 3), torch.float32, 41)
    torch.cuda.synchronize()
    for fn in (ks.temporal_convolution_batched, ks.gaussian_convolution3D_batched):
        n0 = lib.kccot_launch_count()
        with pytest.raises(ValueError, match="2 problems for a batch of 3"):
            fn(x, SmoothingTaps(3, nprob=2).set(1.0))
        with pytest.raises(ValueError, match="2 sigmas for 3 problems"):
            fn(x, [1.0, 2.0])
        with pytest.raises(ValueError, match="radius 4 for a filter of radius 3"):
            fn(x, SmoothingTaps(4, nprob=3).set(1.0))
        with pytest.raises(ValueError, match="None problems"):
            fn(x, SmoothingTaps(3).set(1.0))
        with pytest.raises(ValueError, match="weights are on cpu"):
            fn(x, SmoothingTaps(3, device="cpu", nprob=3).set(1.0))
        with pytest.raises(ValueError, match="6 dimensions"):
            fn(x[0], 1.0)
        with pytest.raises(ValueError, match="float32"):
            fn(x.half(), 1.0)
        with pytest.raises(ValueError, match="float32"):
            fn(x.double(), 1.0)
        taps = SmoothingTaps(3, nprob=3).set(1.0)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            y = x + 0.0
            with pytest.raises(ValueError, match="SmoothingTaps"):
                fn(x, [1.0, 2.0, 3.0])
            with pytest.raises(ValueError, match="SmoothingTaps"):
                fn(x, 1.0)
        assert lib.kccot_launch_count() == n0
        del y, taps
    # the single-problem methods still take one video only
    with pytest.raises(ValueError, match="5 dimensions"):
        ks.temporal_convolution(x, 1.0)
