"""bf16 videos in the mixed Sinkhorn loss.  Needs a B200: `pytest -m gpu`.

Contract (include/kccot.h, kccot_mixed_loss_*_bf16): for bf16 f_real / f_fake the mixed loss gives EXACTLY what the
fp32 call gives on f_real.float() / f_fake.float(): loss, terms and the h / m gradients bit for bit, the video
gradients equal to the fp32 gradient rounded to nearest even.  It holds on the native path (bf16 tensor-core kernels:
B <= 64, B % 8 == 0, K % 8 == 0, K >= 128) and on the widened path (every other shape, and PATH_SIMT).
"""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from kccotgan_b200.synthetic import CONFIGS, GRAD_NAMES, INPUT_ORDER, make_inputs

pytestmark = pytest.mark.gpu

S = 1.0 / 15.0
BF = torch.bfloat16


@pytest.fixture(scope="module", autouse=True)
def _device():
    from kccotgan_b200 import _lib
    assert _lib.load().kccot_device_check() == 0, _lib.last_error()


@pytest.fixture(autouse=True)
def _reset_path():
    from kccotgan_b200 import functional
    functional.set_path("auto")
    yield
    functional.set_path("auto")


def _cfg(name):
    return {k: v for k, v in CONFIGS[name].items() if k not in ("nprob", "ctx")}


def _inputs(kind="uniform", seed=1, **shape):
    """bf16 videos (drawn in fp32, rounded) and fp32 h / m on the GPU"""
    d = make_inputs(J=8, kind=kind, seed=seed, device="cuda", **shape)
    d["real"], d["fake"] = d["real"].to(BF), d["fake"].to(BF)
    return d


def _run(inp, video_dtype, ctx_frames=0, want_real=True):
    """-> (loss, terms, grads) of sinkhorn_loss_terms (or the shared-context entry) with the videos cast to video_dtype"""
    from kccotgan_b200 import gan_utils
    leaves = [inp[k].detach().clone() for k in INPUT_ORDER]
    leaves[0], leaves[1] = leaves[0].to(video_dtype), leaves[1].to(video_dtype)
    for i, t in enumerate(leaves):
        t.requires_grad_(i != 0 or want_real)
    r, f, hf, mr, hr, mf = leaves
    if ctx_frames:
        loss, terms = gan_utils.compute_sinkhorn_loss_shared_context(r, f, S, hf, mr, hr, mf, ctx_frames)
    else:
        loss, terms = gan_utils.sinkhorn_loss_terms(r, f, S, hf, mr, hr, mf)
    want = [t for t in leaves if t.requires_grad]
    g = torch.autograd.grad(loss, want)
    grads = dict(zip([n for n, t in zip(GRAD_NAMES, leaves) if t.requires_grad], g))
    torch.cuda.synchronize()
    return loss.detach(), terms.detach(), grads


def _assert_contract(inp, ctx_frames=0):
    loss16, terms16, g16 = _run(inp, BF, ctx_frames)
    loss32, terms32, g32 = _run(inp, torch.float32, ctx_frames)
    assert torch.equal(loss16, loss32), (float(loss16), float(loss32))
    assert torch.equal(terms16, terms32), (terms16, terms32)
    for n in ("h_fake", "m_real", "h_real", "m_fake"):
        assert g16[n].dtype == torch.float32 and torch.equal(g16[n], g32[n]), n
    for n in ("f_real", "f_fake"):
        assert g16[n].dtype == BF, n
        want = g32[n].to(BF)
        if not torch.equal(g16[n], want):
            diff = (g16[n].view(torch.int16).int() - want.view(torch.int16).int()).abs()
            pytest.fail(f"{n}: {int((diff != 0).sum())} elements differ, max {int(diff.max())} bf16 ulps")
    return g16


# ---------------------------------------------------------------------------------------------
# native path
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,kind", [("cfg1_mmnist", "uniform"), ("cfg1_mmnist", "video"),
                                       ("cfg2_mazes", "uniform"), ("cfg2_mazes", "video")])
def test_native_bit_exact_full_size(name, kind):
    _assert_contract(_inputs(kind, **_cfg(name)))


def test_native_shared_context():
    c = _cfg("cfg2_mazes")
    ctx = CONFIGS["cfg2_mazes"]["ctx"]
    g16 = _assert_contract(_inputs("video", ctx=ctx, **c), ctx_frames=ctx)
    assert not g16["f_fake"][:, :, :ctx].any()


def test_native_batched_config4_shape():
    from kccotgan_b200 import gan_utils
    c = _cfg("cfg4_batched")
    P = 16
    sets = [make_inputs(J=8, kind="uniform", seed=7 + q, device="cuda", **c) for q in range(P)]
    stacked = {k: torch.stack([d[k] for d in sets]) for k in INPUT_ORDER}
    stacked["real"], stacked["fake"] = stacked["real"].to(BF), stacked["fake"].to(BF)
    out = {}
    for dt in (BF, torch.float32):
        leaves = [stacked[k].detach().clone() for k in INPUT_ORDER]
        leaves[0], leaves[1] = leaves[0].to(dt), leaves[1].to(dt)
        for t in leaves:
            t.requires_grad_(True)
        loss = gan_utils.compute_sinkhorn_loss_batched(*leaves[:2], S, *leaves[2:])
        g = torch.autograd.grad(loss.sum(), leaves)
        out[dt] = (loss.detach(), g)
    assert torch.equal(out[BF][0], out[torch.float32][0])
    for n, a, b in zip(GRAD_NAMES, out[BF][1], out[torch.float32][1]):
        if n in ("f_real", "f_fake"):
            assert a.dtype == BF and torch.equal(a, b.to(BF)), n
        else:
            assert torch.equal(a, b), n


def test_native_keeps_no_fp32_copies():
    from kccotgan_b200 import _lib
    from kccotgan_b200.functional import MixedLossFn
    inp = _inputs("uniform", **_cfg("cfg2_mazes"))
    r, f = inp["real"].requires_grad_(True), inp["fake"].requires_grad_(True)
    loss, _ = MixedLossFn.apply(r, f, inp["h_fake"], inp["m_real"], inp["h_real"], inp["m_fake"], S, 1.0, 100)
    saved = loss.grad_fn.saved_tensors
    assert saved[0].dtype == BF and saved[1].dtype == BF
    lib = _lib.load()
    B, K = r.shape[0], r[0].numel()
    for b, k in ((B, K), (32, 81920), (8, 128)):
        assert lib.kccot_mixed_loss_workspace_bytes_bf16(1, b, k, 100, 0) == lib.kccot_mixed_loss_workspace_bytes(1, b, k, 100)


# ---------------------------------------------------------------------------------------------
# widened path
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,path", [
    (dict(B=30, T=6, H=16, W=16, C=1), "auto"),        # B % 8 != 0
    (dict(B=16, T=5, H=6, W=10, C=1), "auto"),         # K = 300: K % 8 == 4
    (dict(B=32, T=8, H=16, W=16, C=1), "simt"),        # PATH_SIMT
    (dict(B=128, T=4, H=16, W=16, C=1), "auto"),       # B > 64: large-batch kernels
])
def test_widened_bit_exact(shape, path):
    from kccotgan_b200 import functional
    functional.set_path(path)
    _assert_contract(_inputs("uniform", **shape))


# ---------------------------------------------------------------------------------------------
# against the fp64 oracle on the bf16-rounded inputs
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,T,D", [(32, 10, 256), (64, 6, 512)])
def test_oracle_parity(B, T, D):
    from kccotgan_b200 import gan_utils
    from oracle import closed_form as cf
    g = torch.Generator().manual_seed(B + T)
    real = torch.rand((B, T, D), generator=g).to(BF)
    fake = (real.float() + 0.3 * torch.rand((B, T, D), generator=g)).clamp_(0, 1).to(BF)
    hm = [torch.sigmoid(torch.randn((B, T, 8), generator=g)) for _ in range(4)]
    leaves = [t.cuda().requires_grad_(True) for t in (real, fake, *hm)]
    loss, terms = gan_utils.sinkhorn_loss_terms(*leaves[:2], S, *leaves[2:])
    grads = torch.autograd.grad(loss, leaves)
    a = [t.float().numpy().astype(np.float64) for t in (real, fake, *hm)]
    ref, gref, det = cf.compute_sinkhorn_loss(a[0], a[1], S, 0.8, 100, a[2], a[3], a[4], a[5], grad=True)
    ref_terms = np.array([det["loss_xy"], det["loss_xx"], det["loss_yy"]])
    scale = np.abs(ref_terms).max()
    assert np.abs(terms.cpu().numpy() - ref_terms).max() <= 1e-4 * scale
    assert abs(float(loss) - ref) <= 1e-4 * scale
    for n, t in zip(GRAD_NAMES, grads):
        e = rel_l2(t.float().cpu().numpy().astype(np.float64), gref[n])
        assert e < (4e-3 if n in ("f_real", "f_fake") else 1e-4), (n, e)


# ---------------------------------------------------------------------------------------------
# dtypes
# ---------------------------------------------------------------------------------------------
def test_mixed_video_dtypes_equal_fp32():
    from kccotgan_b200 import gan_utils
    inp = _inputs("uniform", **_cfg("cfg1_mmnist"))
    res = {}
    for fake_dt in (BF, torch.float32):
        leaves = [inp[k].detach().clone() for k in INPUT_ORDER]
        leaves[0], leaves[1] = leaves[0].float(), leaves[1].to(fake_dt)
        for t in leaves:
            t.requires_grad_(True)
        loss = gan_utils.compute_sinkhorn_loss(*leaves[:2], S, 0.8, 100, *leaves[2:])
        res[fake_dt] = (loss.detach(), torch.autograd.grad(loss, leaves))
    assert torch.equal(res[BF][0], res[torch.float32][0])
    for n, a, b in zip(GRAD_NAMES, res[BF][1], res[torch.float32][1]):
        if n == "f_fake":
            assert a.dtype == BF and torch.equal(a, b.to(BF))
        else:
            assert a.dtype == torch.float32 and torch.equal(a, b), n


def test_bf16_h_m_and_misaligned_views():
    from kccotgan_b200 import gan_utils
    inp = _inputs("uniform", B=16, T=4, H=8, W=8, C=2)
    # misaligned bf16 views (storage offset of one element) are cloned before the call
    base = [torch.empty(inp[k].numel() + 8, dtype=BF, device="cuda") for k in ("real", "fake")]
    views = []
    for b, k in zip(base, ("real", "fake")):
        v = b[1:1 + inp[k].numel()].view(inp[k].shape)
        v.copy_(inp[k])
        views.append(v.detach().requires_grad_(True))          # same storage offset: data_ptr % 16 == 2
    hm = [inp[k].to(BF).requires_grad_(True) for k in ("h_fake", "m_real", "h_real", "m_fake")]
    loss = gan_utils.compute_sinkhorn_loss(*views, S, 0.8, 100, *hm)
    g = torch.autograd.grad(loss, [*views, *hm])
    assert [t.dtype for t in g] == [BF] * 6
    # bf16 h / m are widened: the same as the fp32 call on the rounded h / m
    inp2 = dict(inp)
    for k in ("h_fake", "m_real", "h_real", "m_fake"):
        inp2[k] = inp[k].to(BF).float()
    ref2, _, g_ref2 = _run(inp2, BF)
    assert torch.equal(loss.detach(), ref2)
    assert torch.equal(g[0], g_ref2["f_real"]) and torch.equal(g[1], g_ref2["f_fake"])
    for t, n in zip(g[2:], ("h_fake", "m_real", "h_real", "m_fake")):
        assert torch.equal(t, g_ref2[n].to(BF)), n


@pytest.mark.parametrize("dt", [torch.float16, torch.float64])
def test_other_dtypes_raise(dt):
    from kccotgan_b200 import gan_utils
    inp = make_inputs(B=8, T=4, H=8, W=8, C=1, device="cuda")
    with pytest.raises(ValueError):
        gan_utils.compute_sinkhorn_loss(inp["real"].to(dt), inp["fake"].to(dt), S, 0.8, 100,
                                        *[inp[k] for k in INPUT_ORDER[2:]])


# ---------------------------------------------------------------------------------------------
# CUDA graphs
# ---------------------------------------------------------------------------------------------
def test_graphed_bf16_and_lanes():
    from kccotgan_b200.graphed import EvaluationLanes, GraphedSinkhornLoss
    c = _cfg("cfg2_mazes")
    sets = [_inputs("uniform", seed=40 + j, **c) for j in range(8)]
    eager = [_run(d, BF, want_real=False) for d in sets]
    evs = [GraphedSinkhornLoss(*[d[k].clone() for k in INPUT_ORDER], S, adopt=True) for d in sets]
    for ev, (loss, _, grads) in zip(evs, eager):
        ev.step()
        torch.cuda.synchronize()
        assert torch.equal(ev.loss.detach(), loss)
        assert ev.grads["fake"].dtype == BF and torch.equal(ev.grads["fake"], grads["f_fake"])
        for n in ("h_fake", "m_real", "h_real", "m_fake"):
            assert torch.equal(ev.grads[n], grads[n]), n
    serial = [(ev.loss.detach().clone(), {k: v.clone() for k, v in ev.grads.items()}) for ev in evs]
    lanes = EvaluationLanes(evs)
    lanes.fork()
    for j in range(len(lanes)):
        lanes.submit(j)
    lanes.join()
    torch.cuda.synchronize()
    for ev, (loss, grads) in zip(evs, serial):
        assert torch.equal(ev.loss.detach(), loss)
        for k, v in grads.items():
            assert torch.equal(ev.grads[k], v), k
