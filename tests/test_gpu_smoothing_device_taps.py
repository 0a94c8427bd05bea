"""Gaussian smoothing with its weights in device memory (data_utils.SmoothingTaps, kccot_smooth_*_dev).  Needs a B200:
`pytest -m gpu`.

Contract: for the same weight values the *_dev entries compute what the host-weight entries compute — out, maxval and
the bf16 tie mask bit for bit, gx bit for bit outside the adjoint stencil of the tied maxima (inside it both sum
S = sum(gout * out) with atomics, in an order that varies from run to run).  SmoothFn snapshots the weights in the
forward, so a .set() before the backward does not reach the gradient, and a CUDA graph captured with a SmoothingTaps
filters with the weights of the last .set() before each replay: kernel_train.py's annealed sigma in a graph.
"""
import numpy as np
import pytest
import torch

from test_gpu_bf16_smoothing import _support, _unpack

pytestmark = pytest.mark.gpu

BF = torch.bfloat16


@pytest.fixture(scope="module", autouse=True)
def _device():
    from kccotgan_b200 import _lib
    assert _lib.load().kccot_device_check() == 0, _lib.last_error()


def _ks(r=3):
    from kccotgan_b200.data_utils import KernelSmoothing
    return KernelSmoothing(temporal_kernel_size=2 * r, spatial_kernel_size=2 * r)


def _taps(r, sigma):
    from kccotgan_b200.data_utils import SmoothingTaps
    return SmoothingTaps(r).set(sigma)


def _abi(mode, x, gout, r, sigma, dev):
    """forward and backward through the C ABI, with host weights (dev=False) or the *_dev entries
    -> (out, maxval, tie mask or None, gx)"""
    from kccotgan_b200 import _lib
    from kccotgan_b200.data_utils import KernelSmoothing
    from kccotgan_b200.functional import _ptr, _stream, _taps as host_taps
    lib = _lib.load()
    B, H, T, W, C = x.shape
    bf16 = x.dtype == BF
    if dev:
        wd = _taps(r, sigma).weights
        wargs = (_ptr(wd), r)
    else:
        h = host_taps(tuple(KernelSmoothing._weights(r, sigma)))
        wargs = (*h, None, 0) if mode == 1 else (None, 0, *h)
    sfx = ("_bf16" if bf16 else "") + ("_dev" if dev else "")
    ws = torch.empty(max(256, lib.kccot_smooth_workspace_bytes(mode, B, H, T, W, C)), dtype=torch.uint8, device="cuda")
    out, gx, mx = torch.empty_like(x), torch.empty_like(x), torch.empty(1, device="cuda")
    st = _stream(x.device)
    if bf16:
        ties = torch.full((lib.kccot_smooth_ties_bytes(B, H, T, W, C) // 4,), -1, dtype=torch.int32, device="cuda")
        _lib.call("kccot_smooth_fwd" + sfx, mode, _ptr(x), B, H, T, W, C, *wargs, _ptr(out), _ptr(mx), _ptr(ties),
                  _ptr(ws), ws.numel(), st)
        _lib.call("kccot_smooth_bwd" + sfx, mode, _ptr(gout), _ptr(out), _ptr(mx), _ptr(ties), B, H, T, W, C, *wargs,
                  _ptr(gx), _ptr(ws), ws.numel(), st)
    else:
        ties = None
        _lib.call("kccot_smooth_fwd" + sfx, mode, _ptr(x), B, H, T, W, C, *wargs, _ptr(out), _ptr(mx), _ptr(ws),
                  ws.numel(), st)
        _lib.call("kccot_smooth_bwd" + sfx, mode, _ptr(gout), _ptr(out), _ptr(mx), B, H, T, W, C, *wargs, _ptr(gx),
                  _ptr(ws), ws.numel(), st)
    torch.cuda.synchronize()
    return out, mx, ties, gx


def _assert_grad(mode, r, sigma, tie, got, want):
    """gx equal outside the tie stencil; inside it, within S's run-to-run rounding.  S sums ~10^7 products through one
    atomic per CTA, in an order that changes between runs: at config 3 two calls of the same entry differ there by a few
    1e-6 of the stencil's largest |gx| (the tie term dominates it).  Held to 1e-5 of that in fp32, one bf16 unit in
    bf16."""
    inside = torch.from_numpy(_support(tie.reshape(got.shape), "1d" if mode == 1 else "3d", r, sigma)).cuda()
    assert torch.equal(got[~inside], want[~inside]), (mode, r, tuple(got.shape))
    a, b = got[inside].double(), want[inside].double()
    if a.numel():
        tol = 1e-5 * b.abs().max() if got.dtype == torch.float32 else 2.0 ** -8 * (b.abs() + b.abs().max())
        assert bool(((a - b).abs() <= tol).all()), (mode, r, (a - b).abs().max())


def _check_same(mode, x, r, sigma, seed=0):
    gout = torch.randn(x.shape, generator=torch.Generator().manual_seed(seed)).to(x.dtype).cuda()
    if x.data_ptr() % 16:                                   # keep gout's misalignment like x's
        g = torch.empty(x.numel() + 1, dtype=x.dtype, device="cuda")
        gout = g[1:].view(x.shape).copy_(gout)
    o0, m0, t0, g0 = _abi(mode, x, gout, r, sigma, dev=False)
    o1, m1, t1, g1 = _abi(mode, x, gout, r, sigma, dev=True)
    assert torch.equal(o1, o0) and torch.equal(m1, m0), (mode, r, tuple(x.shape))
    if t0 is not None:
        assert torch.equal(t1, t0)
        tie = _unpack(t0, x.numel())
    else:
        tie = (o0 == 1.0).cpu().numpy().reshape(-1)
    assert tie.any()
    _assert_grad(mode, r, sigma, tie, g1, g0)


def _draw(shape, dtype, seed):
    return torch.rand(shape, generator=torch.Generator().manual_seed(seed)).to(dtype).cuda()


# shapes [B,H,T,W,C] -> the kernels of the T pass (mode 1; mode 3 adds its H and W passes): tile (inner = W*C < 64,
# C = 1 and 3), column with 4 elements per thread (and 8 in bf16 on the large one), column with 1 (inner % 4 != 0)
SHAPES = [(2, 9, 8, 10, 1), (3, 16, 8, 12, 3), (2, 16, 8, 64, 2), (8, 128, 7, 64, 24), (2, 14, 9, 65, 1)]


@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
@pytest.mark.parametrize("r", [1, 3, 6])
@pytest.mark.parametrize("mode", [1, 3])
@pytest.mark.parametrize("shape", SHAPES)
def test_same_numbers_as_host_weights(shape, mode, r, dtype):
    _check_same(mode, _draw(shape, dtype, sum(shape) + r), r, 0.5 + r)


@pytest.mark.parametrize("mode", [1, 3])
def test_misaligned_bf16_view(mode):
    """a storage offset of one element (2 bytes): the bf16 kernels take their one-element paths"""
    shape = (2, 16, 8, 16, 3)
    x = _draw((int(np.prod(shape)) + 1,), BF, 11)
    xv = x[1:].view(shape)
    assert xv.data_ptr() % 16 == 2
    _check_same(mode, xv, 3, 3.0)


@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
def test_config3_full_size(dtype):
    """[64, 64, 12, 64, 3], the BAIR shape of config 3, temporal smoothing"""
    from kccotgan_b200.synthetic import CONFIGS
    c = CONFIGS["cfg3_bair"]
    _check_same(1, _draw((c["B"], c["H"], c["T"], c["W"], c["C"]), dtype, 3), 3, 5.0)


def _fwd_bwd(fn, x, gout, sigma):
    xl = x.detach().requires_grad_(True)
    out = fn(xl, sigma)
    gx, = torch.autograd.grad(out, xl, gout)
    return out.detach(), gx


def _fns(ks):
    return ((1, ks.temporal_convolution, ks.temporal_radius), (3, ks.gaussian_convolution3D, ks.spatial_radius))


def _assert_eager_equal(mode, r, sigma, out, gx, out_ref, gx_ref):
    assert torch.equal(out, out_ref), (mode, sigma)
    tie = (out_ref.float() == 1.0).cpu().numpy().reshape(-1)
    if out.dtype == BF:                 # (the bf16 output cannot tell ties from near-ties: use a generous support)
        tie = (out_ref.float() >= 1.0 - 2.0 ** -8).cpu().numpy().reshape(-1)
    _assert_grad(mode, r, sigma, tie, gx, gx_ref)


@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
def test_backward_uses_the_forward_weights(dtype):
    """forward at sigma = 5, .set(0.7), backward: the gradient is the sigma = 5 one"""
    ks = _ks()
    x = _draw((2, 16, 8, 16, 3), dtype, 7)
    gout = torch.randn(x.shape, generator=torch.Generator().manual_seed(8)).to(dtype).cuda()
    for mode, fn, r in _fns(ks):
        taps = _taps(r, 5.0)
        xl = x.detach().requires_grad_(True)
        out = fn(xl, taps)
        taps.set(0.7)
        gx, = torch.autograd.grad(out, xl, gout)
        out_ref, gx_ref = _fwd_bwd(fn, x, gout, 5.0)
        torch.cuda.synchronize()
        _assert_eager_equal(mode, r, 5.0, out.detach(), gx, out_ref, gx_ref)


@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
def test_graph_follows_set(dtype):
    """forward + backward of both smoothings captured once with a SmoothingTaps; every replay after a .set(sigma) equals
    the eager float-sigma call at that sigma"""
    ks = _ks()
    x = _draw((2, 16, 8, 16, 3), dtype, 21)
    gout = torch.randn(x.shape, generator=torch.Generator().manual_seed(22)).to(dtype).cuda()
    taps = _taps(3, 5.0)
    xl = x.detach().requires_grad_(True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                               # warm-up outside the capture
        for _, fn, _ in _fns(ks):
            torch.autograd.grad(fn(xl, taps), xl, gout)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        res = []
        for _, fn, _ in _fns(ks):
            out = fn(xl, taps)
            gx, = torch.autograd.grad(out, xl, gout)
            res.append((out.detach(), gx))
    graph.replay()
    torch.cuda.synchronize()
    at_capture = [o.clone() for o, _ in res]
    for sigma in [ks.annealing_sigma(5.0, s) for s in (0, 1, 500, 5000, 12345)] + [0.8]:
        taps.set(sigma)
        graph.replay()
        torch.cuda.synchronize()
        for (mode, fn, r), (out, gx), out0 in zip(_fns(ks), res, at_capture):
            out_ref, gx_ref = _fwd_bwd(fn, x, gout, sigma)
            torch.cuda.synchronize()
            _assert_eager_equal(mode, r, sigma, out, gx, out_ref, gx_ref)
            if sigma == 0.8:
                assert not torch.equal(out, out0), mode          # the replay really filtered with other weights


@pytest.mark.parametrize("kernel", ["1d", "3d"])
def test_graphed_training_iteration_with_annealed_sigma(kernel):
    """GraphedTrainingIteration.step(sigma_i) follows the eager capturable closures on the same sigma sequence, and
    step() replays the constructor's sigma"""
    from kccotgan_b200.data_utils import KernelSmoothing
    from kccotgan_b200.train_step import GraphedTrainingIteration, StubDiscriminator, StubGenerator, make_training_steps
    B, H, T, ctx, W, C = 8, 16, 8, 2, 16, 3
    x = [torch.rand(B, H, T, W, C, device="cuda", generator=torch.Generator(device="cuda").manual_seed(70 + i))
         for i in range(5)]
    sigmas = [KernelSmoothing().annealing_sigma(5.0, 1000 * i) for i in range(4)] + [5.0]

    def build():
        torch.manual_seed(9)
        gen = StubGenerator(T - ctx, C).cuda()
        dh, dm = StubDiscriminator(H, W, C).cuda(), StubDiscriminator(H, W, C).cuda()
        return gen, dh, dm

    gen, dh, dm = build()
    disc_step, gen_step = make_training_steps(gen, dh, dm, B, kernel_choice=kernel, gen_lr=1e-2, disc_lr=1e-2,
                                              capturable=True)
    warm = 2
    torch.manual_seed(123)
    for _ in range(warm):
        disc_step(x[0][:, :, :ctx], x[0][:, :, ctx:], 5.0)
        gen_step(x[0][:, :, :ctx], x[0][:, :, ctx:], 5.0)
    outs = []
    for xi, sigma in zip(x, sigmas):
        pm = disc_step(xi[:, :, :ctx], xi[:, :, ctx:], sigma)
        loss = gen_step(xi[:, :, :ctx], xi[:, :, ctx:], sigma)
        outs.append((float(loss), float(pm)))

    gen2, dh2, dm2 = build()
    torch.manual_seed(123)
    it = GraphedTrainingIteration(gen2, dh2, dm2, x[0][:, :, :ctx], x[0][:, :, ctx:], sigma=5.0, warmup=warm,
                                  kernel_choice=kernel, gen_lr=1e-2, disc_lr=1e-2)
    for i, (xi, sigma) in enumerate(zip(x, sigmas)):
        it.real_in.copy_(xi[:, :, :ctx])
        it.real_pred.copy_(xi[:, :, ctx:])
        loss, pm = it.step(sigma) if i < 4 else it.step()          # the last one: back to the constructor's 5.0
        torch.cuda.synchronize()
        assert np.isfinite(float(loss)) and np.isfinite(float(pm))
        assert abs(float(loss) - outs[i][0]) <= 1e-4 * max(1.0, abs(outs[i][0])), (i, float(loss), outs[i])
        assert abs(float(pm) - outs[i][1]) <= 1e-4 * max(1.0, abs(outs[i][1])), (i, float(pm), outs[i])
    assert torch.equal(it.taps.weights.cpu(), torch.from_numpy(KernelSmoothing._weights(3, 5.0)))


def test_set_does_not_synchronise():
    taps = _taps(3, 5.0)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for step in range(50):
            taps.set(_ks().annealing_sigma(5.0, step))
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.equal(taps.weights.cpu(), torch.from_numpy(_ks()._weights(3, _ks().annealing_sigma(5.0, 49))))
