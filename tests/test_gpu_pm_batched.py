"""Martingale penalty of batched independent problems (gan_utils.scale_invariante_martingale_regularization_batched,
kccot_pm_batched_*).  Needs a B200: `pytest -m gpu`.

Contract: for each problem p of an M [nprob, B, T, J] call, against kccot_pm_fwd / _bwd called on M[p] with upstream
gradient gpm[p], pm[p], stats row p and gM[p] are bit-identical.  A problem with sigma_j = 0 takes the single call's
branch and changes no other problem's numbers.  A bf16 M gives the fp32 numbers of M.float(), its gradient rounded.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_l2

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-4
GRAD_TOL = 1e-4
LAM, S = 1.3, 1.0 / 15.0


@pytest.fixture(scope="module", autouse=True)
def _device():
    from kccotgan_b200 import _lib
    assert _lib.load().kccot_device_check() == 0, _lib.last_error()


def _draw(shape, seed):
    """problems of different location and scale, so that no two share their statistics"""
    g = torch.Generator().manual_seed(seed)
    P = shape[0]
    loc = torch.randn((P, 1, 1, 1), generator=g)
    scale = 0.1 + torch.rand((P, 1, 1, 1), generator=g)
    return (loc + scale * torch.randn(shape, generator=g)).cuda()


def _gpm(P, seed):
    return torch.randn(P, generator=torch.Generator().manual_seed(seed)).cuda()


def _batched_abi(M, gpm):
    """-> (pm [nprob], stats [nprob, 2J + (T-1)J], gM) of kccot_pm_batched_fwd / _bwd"""
    from kccotgan_b200 import _lib
    from kccotgan_b200.functional import _ptr, _stream
    P, B, T, J = M.shape
    pm = torch.full((P,), float("nan"), device="cuda")
    stats = torch.full((P, 2 * J + (T - 1) * J), float("nan"), device="cuda")
    gM = torch.full_like(M, float("nan"))
    st = _stream(M.device)
    _lib.call("kccot_pm_batched_fwd", _ptr(M), P, B, T, J, LAM, S, _ptr(pm), _ptr(stats), st)
    _lib.call("kccot_pm_batched_bwd", _ptr(M), P, B, T, J, LAM, S, _ptr(stats), _ptr(gpm), _ptr(gM), st)
    torch.cuda.synchronize()
    return pm, stats, gM


def _single_abi(M, gpm):
    """the same three from one kccot_pm_fwd / _bwd call per problem"""
    from kccotgan_b200 import _lib
    from kccotgan_b200.functional import _ptr, _stream
    P, B, T, J = M.shape
    pm = torch.full((P,), float("nan"), device="cuda")
    stats = torch.full((P, 2 * J + (T - 1) * J), float("nan"), device="cuda")
    gM = torch.full_like(M, float("nan"))
    st = _stream(M.device)
    for p in range(P):
        _lib.call("kccot_pm_fwd", _ptr(M[p]), B, T, J, LAM, S, _ptr(pm[p:]), _ptr(stats[p]), st)
        _lib.call("kccot_pm_bwd", _ptr(M[p]), B, T, J, LAM, S, _ptr(stats[p]), _ptr(gpm[p:]), _ptr(gM[p]), st)
    torch.cuda.synchronize()
    return pm, stats, gM


def _assert_equal(a, b, what):
    for x, y, name in zip(a, b, ("pm", "stats", "gM")):
        assert torch.equal(x, y), (what, name, (x != y).nonzero()[:5].tolist())


@pytest.mark.parametrize("nprob", [1, 3, 256])
@pytest.mark.parametrize("shape", [(64, 10, 8), (32, 20, 8), (7, 3, 5), (1024, 20, 8)])
def test_same_bits_as_single_calls(shape, nprob):
    M = _draw((nprob, *shape), sum(shape) + nprob)
    gpm = _gpm(nprob, nprob)
    _assert_equal(_batched_abi(M, gpm), _single_abi(M, gpm), (shape, nprob))


def test_python_function_matches_single_calls_and_golden():
    """the two p_M cases of the golden file as two problems of one call: the same bits as the single-problem Python
    function, each within the parity bar of test_pm_small of the reference's own fp64 numbers"""
    from kccotgan_b200 import gan_utils
    g = load_golden("gan_utils_small.npz")
    s = float(g["scaling_coef"])
    M = torch.stack([torch.from_numpy(g["Mx"]), torch.from_numpy(g["My"])]).cuda().requires_grad_(True)
    pm = gan_utils.scale_invariante_martingale_regularization_batched(M, 1.3, s)
    assert pm.shape == (2,) and pm.dtype == torch.float32
    w = torch.tensor([0.7, -1.9], device="cuda")
    gM, = torch.autograd.grad((pm * w).sum(), M)
    for p, tag in enumerate(("a", "b")):
        Mp = M[p].detach().clone().requires_grad_(True)
        pm1 = gan_utils.scale_invariante_martingale_regularization(Mp, 1.3, s)
        g1, = torch.autograd.grad(pm1 * w[p], Mp)
        assert torch.equal(pm[p].detach(), pm1.detach()) and torch.equal(gM[p], g1), tag
        ref = float(g[f"pm_{tag}"])
        assert abs(float(pm[p].detach()) - ref) <= LOSS_TOL * abs(ref), tag
        assert rel_l2(gM[p].cpu().numpy() / float(w[p]), g[f"pm_{tag}_grad"]) < GRAD_TOL, tag


@pytest.mark.parametrize("shape", [(64, 10, 8), (7, 3, 5), (1024, 20, 8)])
def test_fp64_oracle(shape):
    from kccotgan_b200 import gan_utils
    from oracle import closed_form as cf
    P = 3
    M = _draw((P, *shape), 7 + sum(shape)).requires_grad_(True)
    pm = gan_utils.scale_invariante_martingale_regularization_batched(M, LAM, S)
    gM, = torch.autograd.grad(pm.sum(), M)
    for p in range(P):
        ref, gref = cf.martingale_regularization(M[p].detach().cpu().numpy().astype(np.float64), LAM, S, grad=True)
        assert abs(float(pm[p].detach()) - ref) <= LOSS_TOL * abs(ref), (shape, p, float(pm[p].detach()), ref)
        assert rel_l2(gM[p].cpu().numpy(), gref) < GRAD_TOL, (shape, p)


def test_constant_problem_stays_in_its_slot():
    """a constant M (sigma_j = 0 for every j) as problem 2 of 5: its numbers are those of its own single call (zero
    penalty and gradient, the sd > 0 branch not taken), and problems 0, 1, 3, 4 are bit-identical to a batch of the
    four without it"""
    M = _draw((5, 64, 10, 8), 3)
    M[2] = 0.375
    gpm = _gpm(5, 4)
    out = _batched_abi(M, gpm)
    one = _single_abi(M[2:3].contiguous(), gpm[2:3].contiguous())
    _assert_equal([t[2:3] for t in out], one, "constant problem")
    assert float(out[0][2]) == 0.0 and not out[2][2].any()
    assert torch.equal(out[1][2, 8:16], torch.zeros(8, device="cuda"))            # sigma_j row of the stats
    keep = [0, 1, 3, 4]
    four = _batched_abi(M[keep].contiguous(), gpm[keep].contiguous())
    _assert_equal([t[keep] for t in out], four, "neighbours")
    # and one column j constant in one problem: only that column takes the branch
    M2 = _draw((3, 64, 10, 8), 5)
    M2[1, :, :, 6] = -2.0
    gpm2 = _gpm(3, 6)
    out2 = _batched_abi(M2, gpm2)
    _assert_equal(out2, _single_abi(M2, gpm2), "one constant column")
    assert float(out2[1][1, 8 + 6]) == 0.0 and torch.isfinite(out2[2]).all()


def test_bf16_is_the_widened_fp32_call():
    from kccotgan_b200 import gan_utils
    Mb = _draw((5, 64, 10, 8), 9).to(torch.bfloat16).requires_grad_(True)
    Mf = Mb.detach().float().requires_grad_(True)
    w = _gpm(5, 10)
    pb = gan_utils.scale_invariante_martingale_regularization_batched(Mb, LAM, S)
    pf = gan_utils.scale_invariante_martingale_regularization_batched(Mf, LAM, S)
    assert pb.dtype == torch.float32 and torch.equal(pb, pf)
    gb, = torch.autograd.grad((pb * w).sum(), Mb)
    gf, = torch.autograd.grad((pf * w).sum(), Mf)
    assert gb.dtype == torch.bfloat16 and torch.equal(gb, gf.to(torch.bfloat16))


def _objective(leaves):
    """the batched discriminator objective of kernel_train.py:249-250, per problem -loss + p_M(m_real)"""
    from kccotgan_b200 import gan_utils
    real, fake, h_fake, m_real, h_real, m_fake = leaves
    losses = gan_utils.compute_sinkhorn_loss_batched(real, fake, S, h_fake, m_real, h_real, m_fake)
    return (-losses + gan_utils.scale_invariante_martingale_regularization_batched(m_real, LAM, S)).sum()


def _inputs(P, B, H, T, W, C, J, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    vids = [torch.rand((P, B, H, T, W, C), generator=g, device="cuda") for _ in range(2)]
    hm = [torch.sigmoid(torch.randn((P, B, T, J), generator=g, device="cuda")) for _ in range(4)]
    return vids + hm


def test_discriminator_objective_in_a_cuda_graph():
    """forward and autograd.grad w.r.t. m_real, h_real, h_fake, m_fake captured once; replays on new inputs copied into
    the static buffers equal the eager call"""
    P, B, H, T, W, C, J = 3, 64, 8, 10, 8, 1, 8
    static = [t.requires_grad_(True) for t in _inputs(P, B, H, T, W, C, J, 1)]
    wrt = [static[3], static[4], static[2], static[5]]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                                # warm-up outside the capture
        for _ in range(2):
            torch.autograd.grad(_objective(static), wrt)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        obj = _objective(static)
        grads = torch.autograd.grad(obj, wrt)
    for seed in (2, 3):
        new = _inputs(P, B, H, T, W, C, J, seed)
        with torch.no_grad():
            for dst, src in zip(static, new):
                dst.copy_(src)
        graph.replay()
        torch.cuda.synchronize()
        leaves = [t.clone().requires_grad_(True) for t in new]
        obj_ref = _objective(leaves)
        ref = torch.autograd.grad(obj_ref, [leaves[3], leaves[4], leaves[2], leaves[5]])
        assert torch.equal(obj, obj_ref.detach()), seed
        for a, b, n in zip(grads, ref, ("m_real", "h_real", "h_fake", "m_fake")):
            assert torch.equal(a, b), (seed, n)


def test_config4_discriminator_gradient():
    """256 x [64, 10, 8] with 256 x [64, 32, 10, 32, 1] videos: d/dm_real of sum_p (-loss_p + p_M(m_real_p)) through
    the batched calls against the loop of single-problem calls, within the parity bar for every problem"""
    from kccotgan_b200 import gan_utils
    from kccotgan_b200.synthetic import CONFIGS
    c = CONFIGS["cfg4_batched"]
    P, B, H, T, W, C, J = c["nprob"], c["B"], c["H"], c["T"], c["W"], c["C"], 8
    leaves = _inputs(P, B, H, T, W, C, J, 40)
    leaves[3].requires_grad_(True)
    g, = torch.autograd.grad(_objective(leaves), leaves[3])
    real, fake, h_fake, m_real, h_real, m_fake = leaves
    m_real = m_real.detach().clone().requires_grad_(True)
    obj = sum(-gan_utils.compute_sinkhorn_loss(real[p], fake[p], S, 1.0, 100, h_fake[p], m_real[p], h_real[p],
                                               m_fake[p], video=True)
              + gan_utils.scale_invariante_martingale_regularization(m_real[p], LAM, S) for p in range(P))
    g1, = torch.autograd.grad(obj, m_real)
    for p in range(P):
        e = rel_l2(g[p].cpu().numpy(), g1[p].cpu().numpy())
        assert e < GRAD_TOL, (p, e)


def test_python_errors():
    from kccotgan_b200 import _lib, gan_utils
    f = gan_utils.scale_invariante_martingale_regularization_batched
    M = _draw((3, 8, 5, 2), 0)
    torch.cuda.synchronize()
    n0 = _lib.load().kccot_launch_count()
    with pytest.raises(ValueError, match="4 dimensions"):
        f(M[0], 1.0, 0.1)
    with pytest.raises(ValueError, match="4 dimensions"):
        f(M.unsqueeze(0), 1.0, 0.1)
    with pytest.raises(ValueError, match="CUDA"):
        f(M.cpu(), 1.0, 0.1)
    with pytest.raises(ValueError, match="float32"):
        f(M.double(), 1.0, 0.1)
    with pytest.raises(ValueError, match="float32"):
        f(M.half(), 1.0, 0.1)
    with pytest.raises(ValueError, match="2 time steps"):
        f(M[:, :, :1], 1.0, 0.1)
    with pytest.raises(ValueError, match="nprob"):
        f(torch.zeros((65536, 1, 2, 1), device="cuda"), 1.0, 0.1)
    assert _lib.load().kccot_launch_count() == n0
    # the single-problem function still takes fp32 [B, T, J] only
    with pytest.raises(ValueError, match="3 dimensions"):
        gan_utils.scale_invariante_martingale_regularization(M, 1.0, 0.1)
    with pytest.raises(ValueError, match="float32"):
        gan_utils.scale_invariante_martingale_regularization(M[0].to(torch.bfloat16), 1.0, 0.1)
