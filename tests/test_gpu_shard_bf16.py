"""bf16 videos in the row-sharded mixed loss on one GPU (world = 1).  Needs a B200: `pytest -m gpu`.

Contract (include/kccot.h, kccot_shard_cost_*_bf16): ShardedMixedLoss on bf16 videos gives exactly what it gives on
the fp32 videos widened from them: loss, terms and the h / m gradients bit for bit, the `fake` gradient rows the fp32
rows rounded to nearest even; no fp32 copy of a video is made.  Other dtypes are rejected before any launch.
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
# (B, T, H, W, C): K = 4*16*16 (K % 8 == 0), 5*6*10 = 300 (K % 8 != 0), 3*5*7 = 105 (odd K: scalar loads and stores)
SHAPES = [(256, 4, 16, 16, 1), (128, 5, 6, 10, 1), (96, 3, 5, 7, 1)]


@pytest.fixture(scope="module", autouse=True)
def _device():
    from kccotgan_b200 import _lib
    assert _lib.load().kccot_device_check() == 0, _lib.last_error()


def _inputs(B, T, H, W, C, seed=1):
    """bf16 videos (drawn in fp32, rounded) and fp32 h / m on the GPU"""
    d = make_inputs(B, T, H, W, C, J=8, kind="uniform", seed=seed, device="cuda")
    d["real"], d["fake"] = d["real"].to(BF), d["fake"].to(BF)
    return d


def _loss(B, T, H, W, C):
    from kccotgan_b200.sharded import ShardedMixedLoss
    return ShardedMixedLoss(B, T * H * W * C, T, 8, S, device=torch.device("cuda", 0))


def _run(sm, t):
    loss, terms = sm.forward(*t)
    g = sm.backward(1.0)
    torch.cuda.synchronize()
    return loss.clone(), terms.clone(), g


def _widened(inp):
    return [inp[k].float() for k in NAMES]


def _assert_same(r16, r32, dtypes=None):
    """r16 equals r32 with each gradient rounded to the dtype its input had"""
    (l16, t16, g16), (l32, t32, g32) = r16, r32
    assert torch.equal(l16, l32), (float(l16), float(l32))
    assert torch.equal(t16, t32), (t16, t32)
    dtypes = dtypes or {"fake": BF}
    for n in ("fake",) + HM:
        want = g32[n].to(dtypes.get(n, torch.float32))
        assert g16[n].dtype == want.dtype, (n, g16[n].dtype)
        if not torch.equal(g16[n], want):
            a, b = g16[n].float(), want.float()
            pytest.fail(f"{n}: {int((a != b).sum())} of {a.numel()} elements differ")


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_bit_exact_against_widened_fp32(shape):
    inp = _inputs(*shape)
    sm = _loss(*shape)
    r16 = _run(sm, [inp[k] for k in NAMES])
    r32 = _run(sm, _widened(inp))
    _assert_same(r16, r32)
    assert r16[2]["fake"].shape == inp["fake"].shape


@pytest.mark.parametrize("shape", SHAPES[:2], ids=lambda s: "x".join(map(str, s)))
def test_oracle_parity(shape):
    from oracle import closed_form as cf
    inp = _inputs(*shape)
    loss, terms, g = _run(_loss(*shape), [inp[k] for k in NAMES])
    npin = [inp[k].double().cpu().numpy() for k in NAMES]
    ref, gref, det = cf.compute_sinkhorn_loss(npin[0], npin[1], S, 0.8, 100, *npin[2:], video=True, grad=True)
    ref_terms = np.array([det["loss_xy"], det["loss_xx"], det["loss_yy"]])
    scale = np.abs(ref_terms).max()
    assert np.abs(terms.double().cpu().numpy() - ref_terms).max() <= 1e-4 * scale
    assert abs(float(loss) - ref) <= 1e-4 * scale
    for k, n, tol in (("fake", "f_fake", 4e-3), ("h_fake", "h_fake", 1e-4), ("m_real", "m_real", 1e-4),
                      ("h_real", "h_real", 1e-4), ("m_fake", "m_fake", 1e-4)):
        e = rel_l2(g[k].double().cpu().numpy().reshape(gref[n].shape), gref[n])
        assert e <= tol, (k, e)


def test_mixed_dtypes_widen_exactly():
    shape = SHAPES[1]
    inp = _inputs(*shape)
    sm = _loss(*shape)
    r32 = _run(sm, _widened(inp))
    # bf16 real next to an fp32 fake: both widened, the fake gradient stays fp32
    t = [inp["real"], inp["fake"].float()] + [inp[k] for k in HM]
    _assert_same(_run(sm, t), r32, {"fake": torch.float32})
    # bf16 h / m (with bf16 videos): h and m widened, every gradient in its input's dtype
    hm16 = {k: inp[k].to(BF) for k in HM}
    t = [inp["real"], inp["fake"]] + [hm16[k] for k in HM]
    w = _widened(inp)[:2] + [hm16[k].float() for k in HM]
    _assert_same(_run(sm, t), _run(sm, w), {"fake": BF, **{k: BF for k in HM}})


def test_no_fp32_copy_of_the_videos():
    shape = SHAPES[0]
    inp = _inputs(*shape)
    sm = _loss(*shape)
    t16 = [inp[k] for k in NAMES]
    t32 = _widened(inp)
    peaks = {}
    for name, t in (("fp32", t32), ("bf16", t16), ("fp32", t32), ("bf16", t16)):
        _run(sm, t)                                               # warm: every buffer of this dtype allocated once
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        r = _run(sm, t)
        peaks[name] = torch.cuda.max_memory_allocated() - base
        del r
    B, K = shape[0], shape[1] * shape[2] * shape[3] * shape[4]
    # a widening copy of both videos would add 8 B K bytes to the bf16 peak; the bf16 fake rows save 2 B K
    assert peaks["bf16"] <= peaks["fp32"], (peaks, 8 * B * K)


def test_misaligned_view_gives_the_aligned_result():
    shape = SHAPES[1]
    inp = _inputs(*shape)
    sm = _loss(*shape)
    ref = _run(sm, [inp[k] for k in NAMES])
    views = []
    for k in ("real", "fake"):
        buf = torch.empty(inp[k].numel() + 1, dtype=BF, device="cuda")
        v = buf[1:].view(inp[k].shape)
        v.copy_(inp[k])
        assert v.data_ptr() % 16 != 0
        views.append(v)
    got = _run(sm, views + [inp[k] for k in HM])
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    for n in ("fake",) + HM:
        assert torch.equal(got[2][n], ref[2][n]), n


def test_rejected_inputs_raise_before_any_launch():
    from kccotgan_b200 import _lib
    shape = SHAPES[2]
    inp = _inputs(*shape)
    sm = _loss(*shape)
    hm = [inp[k] for k in HM]
    cases = {
        "fp16 videos": [inp["real"].half(), inp["fake"].half()] + hm,
        "fp64 videos": [inp["real"].double(), inp["fake"].double()] + hm,
        "CPU videos": [inp["real"].cpu(), inp["fake"].cpu()] + hm,
        "fp16 h": [inp["real"], inp["fake"], hm[0].half()] + hm[1:],
        "h of the wrong shape": [inp["real"], inp["fake"], hm[0][:, :-1]] + hm[1:],
    }
    torch.cuda.synchronize()
    n0 = _lib.load().kccot_launch_count()
    for name, t in cases.items():
        with pytest.raises(ValueError):
            sm.forward(*t)
    assert _lib.load().kccot_launch_count() == n0
