"""Shared context frames in the row-sharded mixed loss on one GPU (world = 1).  Needs a B200: `pytest -m gpu`.

Contract (include/kccot.h, kccot_shard_cost_*_ctx): with `ctx_frames` > 0, ShardedMixedLoss never reads fake's context
frames and computes their Gram once for the three cost blocks.  On inputs whose first ctx frames agree, the result
equals the plain sharded result within floating-point tolerance and meets the fp64 oracle; the `fake` gradient is that
of the predicted frames and exactly zero on the context frames.  bf16 videos give the hinted fp32 result on the widened
videos, the `fake` rows rounded to nearest even.
"""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from kccotgan_b200.synthetic import make_inputs

pytestmark = pytest.mark.gpu

S = 1.0 / 15.0
BF = torch.bfloat16
NAMES = ("real", "fake", "h_fake", "m_real", "h_real", "m_fake")
HM = ("h_fake", "m_real", "h_real", "m_fake")
GRADS = ("fake",) + HM
# (B, T, H, W, C, ctx): ctx_len 16 (a multiple of 4: vector loads), 20 (not a multiple of 64), 7 with odd K = 105
SHAPES = [(256, 4, 16, 16, 1, 1), (128, 5, 6, 10, 1, 2), (96, 3, 5, 7, 1, 1)]
KINDS = ("uniform", "video")
# Measured on one B200 over the SHAPES x KINDS below: the hinted and the plain sharded results differ by at most
# 4.1e-7 of the largest term (loss 9.6e-7) and 4.1e-6 rel-L2 in a gradient (fake, predicted frames), the size of the
# reordered fp32 sums (the context and predicted parts of each dot product are summed separately).  The bounds leave a
# factor of 5 to 10 and stay 5x inside the oracle bar of 1e-4.
PLAIN_TERMS_TOL, PLAIN_GRAD_TOL = 1e-5, 2e-5
ID = "x".join


@pytest.fixture(scope="module", autouse=True)
def _device():
    from kccotgan_b200 import _lib
    assert _lib.load().kccot_device_check() == 0, _lib.last_error()


def _inputs(B, T, H, W, C, ctx, kind, seed=1):
    d = make_inputs(B, T, H, W, C, J=8, ctx=ctx, kind=kind, seed=seed, device="cuda")
    d["fake"][:, :, :ctx] = d["real"][:, :, :ctx]          # kind="video" already shares them; uniform needs the copy
    return d


def _loss(B, T, H, W, C, ctx, **kw):
    from kccotgan_b200.sharded import ShardedMixedLoss
    return ShardedMixedLoss(B, T * H * W * C, T, 8, S, device=torch.device("cuda", 0), **kw)


def _run(sm, t):
    loss, terms = sm.forward(*t)
    g = sm.backward(1.0)
    torch.cuda.synchronize()
    return loss.clone(), terms.clone(), {k: v.clone() for k, v in g.items()}


def _assert_equal(a, b):
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), (a[1], b[1])
    for n in GRADS:
        if not torch.equal(a[2][n], b[2][n]):
            x, y = a[2][n].float(), b[2][n].float()
            pytest.fail(f"{n}: {int((x != y).sum())} of {x.numel()} elements differ")


_cache = {}


def _hinted(shape, kind):
    """inputs, hinted result and plain result of one case (computed once per module)"""
    key = (shape, kind)
    if key not in _cache:
        inp = _inputs(*shape, kind)
        t = [inp[k] for k in NAMES]
        _cache[key] = (inp, _run(_loss(*shape, ctx_frames=shape[-1]), t), _run(_loss(*shape), t))
    return _cache[key]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: ID(map(str, s)))
def test_no_hint_is_the_plain_call(shape):
    """ctx_frames = 0, and the _ctx entry points with ctx_len = 0, are the plain sharded call bit for bit"""
    from kccotgan_b200.sharded import CudaMixedShardBackend
    B, T, H, W, C, ctx = shape
    inp = _inputs(*shape, "uniform")
    t = [inp[k] for k in NAMES]
    plain = _run(_loss(*shape), t)
    _assert_equal(_run(_loss(*shape, ctx_frames=0), t), plain)
    be = CudaMixedShardBackend(B, T * H * W * C, T, 8, S, 1.0, 100, 0, B, torch.device("cuda", 0), None,
                               ctx=(T * W * C, 0))
    _assert_equal(_run(_loss(*shape, backend=be), t), plain)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: ID(map(str, s)))
def test_oracle_parity(shape, kind):
    from oracle import closed_form as cf
    ctx = shape[-1]
    inp, (loss, terms, g), _ = _hinted(shape, kind)
    npin = [inp[k].double().cpu().numpy() for k in NAMES]
    ref, gref, det = cf.compute_sinkhorn_loss(npin[0], npin[1], S, 0.8, 100, *npin[2:], video=True, grad=True)
    ref_terms = np.array([det["loss_xy"], det["loss_xx"], det["loss_yy"]])
    scale = np.abs(ref_terms).max()
    assert np.abs(terms.double().cpu().numpy() - ref_terms).max() <= 1e-4 * scale
    assert abs(float(loss) - ref) <= 1e-4 * scale
    e = rel_l2(g["fake"][:, :, ctx:].double().cpu().numpy(), gref["f_fake"][:, :, ctx:])
    assert e <= 1e-4, ("fake", e)
    for k in HM:
        e = rel_l2(g[k].double().cpu().numpy(), gref[k])
        assert e <= 1e-4, (k, e)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: ID(map(str, s)))
def test_close_to_the_plain_call(shape, kind):
    ctx = shape[-1]
    _, (loss, terms, g), (loss0, terms0, g0) = _hinted(shape, kind)
    scale = float(terms0.abs().max())
    dterms = float((terms.double() - terms0.double()).abs().max()) / scale
    dloss = abs(float(loss) - float(loss0)) / scale
    dg = {"fake": rel_l2(g["fake"][:, :, ctx:].cpu().numpy(), g0["fake"][:, :, ctx:].cpu().numpy())}
    dg.update({k: rel_l2(g[k].cpu().numpy(), g0[k].cpu().numpy()) for k in HM})
    print(f"{shape} {kind}: terms {dterms:.2e} loss {dloss:.2e} grads " + " ".join(f"{k} {v:.2e}" for k, v in dg.items()))
    assert dterms <= PLAIN_TERMS_TOL and dloss <= PLAIN_TERMS_TOL, (dterms, dloss)
    assert all(v <= PLAIN_GRAD_TOL for v in dg.values()), dg


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: ID(map(str, s)))
def test_context_frames_of_fake_are_not_read(shape):
    ctx = shape[-1]
    inp, ref, _ = _hinted(shape, "uniform")
    fake = inp["fake"].clone()
    fake[:, :, :ctx] = float("nan")
    t = [inp["real"], fake] + [inp[k] for k in HM]
    _assert_equal(_run(_loss(*shape, ctx_frames=ctx), t), ref)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: ID(map(str, s)))
def test_context_gradient_is_zero(shape, kind):
    ctx = shape[-1]
    _, (_, _, g), _ = _hinted(shape, kind)
    assert g["fake"].shape == (shape[0], shape[2], shape[1], shape[3], shape[4])
    assert torch.equal(g["fake"][:, :, :ctx], torch.zeros_like(g["fake"][:, :, :ctx]))
    assert bool((g["fake"][:, :, ctx:] != 0).any())


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: ID(map(str, s)))
def test_bf16_is_the_widened_fp32_call(shape):
    ctx = shape[-1]
    inp = _inputs(*shape, "uniform")
    inp["real"], inp["fake"] = inp["real"].to(BF), inp["fake"].to(BF)
    sm = _loss(*shape, ctx_frames=ctx)
    r16 = _run(sm, [inp[k] for k in NAMES])
    r32 = _run(sm, [inp[k].float() for k in NAMES])
    assert torch.equal(r16[0], r32[0]) and torch.equal(r16[1], r32[1]), (r16[1], r32[1])
    assert r16[2]["fake"].dtype == BF
    assert torch.equal(r16[2]["fake"], r32[2]["fake"].to(BF))
    for k in HM:
        assert torch.equal(r16[2][k], r32[2][k]), k


def test_rejected_shapes():
    shape = SHAPES[0]
    B, T, H, W, C, ctx = shape
    inp = _inputs(*shape, "uniform")
    sm = _loss(*shape, ctx_frames=ctx)
    hm = [inp[k] for k in HM]
    with pytest.raises(ValueError, match="B, H, T, W, C"):
        sm.forward(inp["real"].reshape(B, -1), inp["fake"].reshape(B, -1), *hm)
    with pytest.raises(ValueError, match="B, H, T, W, C"):                        # T on the wrong axis
        sm.forward(inp["real"].transpose(1, 2), inp["fake"].transpose(1, 2), *hm)
