"""T2: the CUDA path (through the C ABI / ctypes) against the golden vectors of the reference's own
source and against the fp64 oracle on the same inputs.  Needs a B200: `pytest -m gpu`.

Tolerances (BASELINE.json north_star: "within 1e-4 relative, in fp32"):
  * each loss term: |term - ref| <= 1e-4 * max(|xy|,|xx|,|yy|)   (the mixed loss 2xy-xx-yy cancels,
    so it is normalised by the largest term, SURVEY.md §7.3);
  * each gradient: rel-L2 <= 1e-4 against the fp64 reference run;
  * cost matrices: max abs error <= 1e-6 * max|C| (what the reference's own fp32 run achieves).
"""
import numpy as np
import pytest
import torch

from conftest import golden_inputs, load_golden, rel_l2
from kccotgan_b200.synthetic import CONFIGS, GRAD_NAMES, INPUT_ORDER, make_inputs

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-4
GRAD_TOL = 1e-4
COST_TOL = 1e-6


@pytest.fixture(scope="module")
def gu():
    from kccotgan_b200 import _lib, gan_utils
    assert _lib.load().kccot_device_check() == 0, _lib.last_error()
    return gan_utils


@pytest.fixture(autouse=True)
def _reset_path():
    from kccotgan_b200 import functional
    functional.set_path("auto")
    yield
    functional.set_path("auto")


def dev(a, grad=False):
    t = torch.as_tensor(np.asarray(a), dtype=torch.float32).cuda()
    return t.requires_grad_(True) if grad else t


def maxrel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / np.abs(b).max())


# ---------------------------------------------------------------------------------------------
# small golden: every gan_utils function
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def small():
    return load_golden("gan_utils_small.npz")


def test_cost_functions_small(gu, small):
    g = small
    s = float(g["scaling_coef"])
    x, y, hy, Mx, hx, My = (dev(g[k]) for k in ("x", "y", "hy", "Mx", "hx", "My"))
    assert maxrel(gu.cost_xy(x, y, s).cpu(), g["cost_xy"]) < COST_TOL
    assert maxrel(gu.modified_cost(x, y, hy, Mx, s).cpu(), g["modified_cost"]) < COST_TOL
    assert maxrel(gu.bi_causal_modified_cost(x, y, hy, Mx, hx, My, s).cpu(), g["bi_causal_modified_cost"]) < COST_TOL
    assert np.allclose(gu.compute_N(Mx[:, :, 0]).cpu().numpy(), g["compute_N"], atol=1e-6)
    cxx = gu.cost_xy(x, x, s).cpu().numpy()
    assert np.all(np.diag(cxx) == 0.0)          # exact zeros as in the reference


@pytest.mark.parametrize("tag,kw", [("default", {}), ("eps0p8", dict(epsilon=0.8)),
                                    ("eps0p3_L20", dict(epsilon=0.3, L=20)), ("L130", dict(L=130)),
                                    ("eps5_L400", dict(epsilon=5.0, L=400))])
def test_compute_sinkhorn_small(gu, small, tag, kw):
    g = small
    s = float(g["scaling_coef"])
    lv = [dev(g[k], grad=True) for k in ("x", "y", "hy", "Mx")]
    c = gu.compute_sinkhorn(lv[0], lv[1], lv[2], lv[3], s, **kw)
    ref = float(g[f"compute_sinkhorn_{tag}"])
    assert abs(float(c) - ref) <= LOSS_TOL * abs(ref)
    grads = torch.autograd.grad(c, lv)
    for n, a in zip(("x", "y", "hy", "Mx"), grads):
        assert rel_l2(a.cpu().numpy(), g[f"compute_sinkhorn_{tag}_grad_{n}"]) < GRAD_TOL, (tag, n)


def test_bicausal_small(gu, small):
    g = small
    s = float(g["scaling_coef"])
    lv = [dev(g[k], grad=True) for k in ("x", "y", "hy", "Mx", "hx", "My")]
    c = gu.compute_sinkhorn(lv[0], lv[1], lv[2], lv[3], s, lv[4], lv[5], epsilon=0.5, L=50, bi_causal=True)
    ref = float(g["compute_sinkhorn_bicausal"])
    assert abs(float(c) - ref) <= LOSS_TOL * abs(ref)
    for n, a in zip(("x", "y", "hy", "Mx", "hx", "My"), torch.autograd.grad(c, lv)):
        assert rel_l2(a.cpu().numpy(), g[f"compute_sinkhorn_bicausal_grad_{n}"]) < GRAD_TOL, n


@pytest.mark.parametrize("tag,kw", [("default", {}), ("eps0p5_L40_Lmin5", dict(epsilon=0.5, L=40, Lmin=5)),
                                    ("eps2_L200_Lmin10", dict(epsilon=2.0, L=200, Lmin=10))])
def test_benchmark_sinkhorn_small(gu, small, tag, kw):
    g = small
    s = float(g["scaling_coef"])
    lv = [dev(g[k], grad=True) for k in ("x", "y")]
    c = gu.benchmark_sinkhorn(lv[0], lv[1], s, **kw)
    ref = float(g[f"benchmark_sinkhorn_{tag}"])
    assert abs(float(c) - ref) <= LOSS_TOL * abs(ref)
    gx, gy = torch.autograd.grad(c, lv)
    assert rel_l2(gx.cpu().numpy(), g[f"benchmark_sinkhorn_{tag}_grad_x"]) < GRAD_TOL
    assert rel_l2(gy.cpu().numpy(), g[f"benchmark_sinkhorn_{tag}_grad_y"]) < GRAD_TOL


def test_eps_l_arguments_ignored(gu, small):
    g = small
    s = float(g["scaling_coef"])
    args = [dev(g[k]) for k in ("x", "y")], [dev(g[k]) for k in ("hy", "Mx", "hx", "My")]
    a = gu.compute_sinkhorn_loss(args[0][0], args[0][1], s, 0.8, 100, *args[1], video=False)
    b = gu.compute_sinkhorn_loss(args[0][0], args[0][1], s, 5.0, 7, *args[1], video=False)
    assert float(a) == float(b)
    assert abs(float(a) - float(g["loss_novideo"])) <= LOSS_TOL * 2.0


def test_pm_small(gu, small):
    g = small
    for tag, key in (("a", "Mx"), ("b", "My")):
        M = dev(g[key], grad=True)
        pm = gu.scale_invariante_martingale_regularization(M, 1.3, float(g["scaling_coef"]))
        ref = float(g[f"pm_{tag}"])
        assert abs(float(pm) - ref) <= LOSS_TOL * abs(ref)
        gm, = torch.autograd.grad(pm, M)
        assert rel_l2(gm.cpu().numpy(), g[f"pm_{tag}_grad"]) < GRAD_TOL


# ---------------------------------------------------------------------------------------------
# mixed loss at the BASELINE configs
# ---------------------------------------------------------------------------------------------
def _run_loss(gu, inp, s):
    leaves = [inp[k].clone().cuda().requires_grad_(True) for k in INPUT_ORDER]
    r, f, hf, mr, hr, mf = leaves
    from kccotgan_b200.gan_utils import sinkhorn_loss_terms
    loss, terms = sinkhorn_loss_terms(r, f, s, hf, mr, hr, mf)
    loss2 = gu.compute_sinkhorn_loss(r, f, s, 0.8, 100, hf, mr, hr, mf, video=True)
    grads = torch.autograd.grad(loss2, leaves)
    assert float(loss) == float(loss2)
    return float(loss2), terms.cpu().numpy().astype(np.float64), [a.cpu().numpy() for a in grads]


@pytest.mark.parametrize("path", ["simt", "tcgen05"])
@pytest.mark.parametrize("kind", ["uniform", "video"])
@pytest.mark.parametrize("cfg", ["cfg1", "cfg2", "cfg3"])
def test_mixed_loss_reduced(gu, cfg, kind, path):
    from kccotgan_b200 import functional
    functional.set_path(path)
    g = load_golden(f"loss_{cfg}_reduced_{kind}.npz")
    s = float(g["scaling_coef"])
    inp = golden_inputs(g)
    loss, terms, grads = _run_loss(gu, inp, s)
    ref_terms = np.array([float(g["loss_xy"]), float(g["loss_xx"]), float(g["loss_yy"])])
    scale = np.abs(ref_terms).max()
    assert np.abs(terms - ref_terms).max() <= LOSS_TOL * scale, (terms, ref_terms)
    assert abs(loss - float(g["loss"])) <= LOSS_TOL * scale
    errs = {n: rel_l2(a, g["grad_" + n]) for n, a in zip(GRAD_NAMES, grads)}
    print(cfg, kind, path, "loss err", abs(loss - float(g["loss"])) / scale, errs)
    for n, e in errs.items():
        assert e < GRAD_TOL, (n, e)


@pytest.mark.parametrize("path", ["simt", "tcgen05"])
@pytest.mark.parametrize("name,kind", [("cfg1_mmnist", "uniform"), ("cfg1_mmnist", "video"), ("cfg2_mazes", "uniform")])
def test_mixed_loss_full_size(gu, name, kind, path):
    from kccotgan_b200 import functional
    functional.set_path(path)
    g = load_golden(f"loss_{name}_full_{kind}.npz")
    s = float(g["scaling_coef"])
    c = {k: v for k, v in CONFIGS[name].items() if k != "nprob"}
    inp = make_inputs(J=8, kind=kind, seed=1, **c)
    # cost matrices first (the numerically delicate part: |C| ~ 1e3, eps = 1)
    from kccotgan_b200.functional import CostFn
    r, f = inp["real"].cuda(), inp["fake"].cuda()
    Cxy = CostFn.apply(r, f, inp["h_fake"].cuda(), inp["m_real"].cuda(), None, None, s).cpu().numpy()
    print(name, kind, path, "C_xy max abs err", np.abs(Cxy - g["C_xy"]).max(), "max |C|", np.abs(g["C_xy"]).max())
    assert maxrel(Cxy, g["C_xy"]) < COST_TOL
    loss, terms, grads = _run_loss(gu, inp, s)
    ref_terms = np.array([float(g["loss_xy"]), float(g["loss_xx"]), float(g["loss_yy"])])
    scale = np.abs(ref_terms).max()
    print("terms", terms, ref_terms, "loss", loss, float(g["loss"]))
    assert np.abs(terms - ref_terms).max() <= LOSS_TOL * scale
    assert abs(loss - float(g["loss"])) <= LOSS_TOL * scale
    for n, a in zip(GRAD_NAMES, grads):
        if ("grad_" + n) in g:
            e = rel_l2(a, g["grad_" + n])
        else:
            st = int(g["grad_" + n + "_stride"])
            flat = a.reshape(-1).astype(np.float64)
            e = rel_l2(flat[::st], g["grad_" + n + "_sample"])
            assert abs(np.linalg.norm(flat) - float(g["grad_" + n + "_norm"])) <= 1e-4 * float(g["grad_" + n + "_norm"])
            probe = np.random.default_rng(7).standard_normal(flat.size)
            # a random projection sees every element: |<err, probe>| ~ ||err|| for a unit-variance probe
            assert abs(flat @ probe - float(g["grad_" + n + "_proj"])) <= 5 * GRAD_TOL * float(g["grad_" + n + "_norm"])
        print("  grad", n, e)
        assert e < GRAD_TOL, (n, e)


# ---------------------------------------------------------------------------------------------
# independent problems in one call (BASELINE config 4's shape of work) and shapes off the fast path,
# through the raw C ABI, every problem against the fp64 oracle
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nprob,B,T,D,path", [
    (5, 16, 5, 96, "tcgen05"),      # batched, W' built by the separate kernel (B % 32 != 0)
    (3, 32, 4, 64, "tcgen05"),      # batched, W' formed inside the gradient kernel
    (4, 64, 3, 40, "auto"),         # batched at the bench's B
    (2, 24, 6, 50, "auto"),         # K % 4 != 0 ... (T*D = 300 is a multiple of 4; B = 24 is off the 32-row W' path)
    (3, 20, 5, 33, "simt"),         # K = 165: CUDA-core kernels only
    (1, 9, 4, 7, "auto"),           # tiny, ragged everything
])
def test_mixed_loss_batched_abi(nprob, B, T, D, path):
    import ctypes
    from kccotgan_b200 import _lib, functional as F
    from oracle import closed_form as cf
    lib = _lib.load()
    J, s, L = 6, 1.0 / 7.0, 100
    K = T * D
    g = torch.Generator().manual_seed(100 * nprob + B)
    real = torch.rand((nprob, B, T, D), generator=g)
    fake = (real + 0.3 * torch.rand((nprob, B, T, D), generator=g)).clamp_(0, 1)
    hm = [torch.sigmoid(torch.randn((nprob, B, T, J), generator=g)) for _ in range(4)]     # h_fake, m_real, h_real, m_fake
    d = [t.cuda().contiguous() for t in (real, fake, *hm)]
    saved = torch.empty(lib.kccot_mixed_loss_saved_bytes(nprob, B, L), dtype=torch.uint8, device="cuda")
    ws = torch.empty(lib.kccot_mixed_loss_workspace_bytes(nprob, B, K, L), dtype=torch.uint8, device="cuda")
    loss = torch.full((nprob,), float("nan"), device="cuda")
    terms = torch.full((nprob, 3), float("nan"), device="cuda")
    flags = {"auto": 0, "simt": 1, "tcgen05": 2}[path]
    st = F._stream(d[0].device)
    p = F._ptr
    _lib.call("kccot_mixed_loss_fwd", p(d[0]), p(d[1]), nprob, B, K, p(d[2]), p(d[3]), p(d[4]), p(d[5]), T, J, s, 1.0, L,
              p(saved), p(loss), p(terms), p(ws), ws.numel(), flags, st)
    gl = torch.linspace(0.5, 1.5, nprob, device="cuda")                 # a different upstream gradient per problem
    grads = [torch.full_like(t, float("nan")) for t in d]
    _lib.call("kccot_mixed_loss_bwd", p(gl), p(d[0]), p(d[1]), nprob, B, K, p(d[2]), p(d[3]), p(d[4]), p(d[5]), T, J, s,
              1.0, L, p(saved), *[p(t) for t in grads], p(ws), ws.numel(), flags, st)
    torch.cuda.synchronize()
    for q in range(nprob):
        a = [t[q].numpy().astype(np.float64) for t in (real, fake, *hm)]
        ref, gref, det = cf.compute_sinkhorn_loss(a[0], a[1], s, 0.8, 100, a[2], a[3], a[4], a[5], grad=True)
        ref_terms = np.array([det["loss_xy"], det["loss_xx"], det["loss_yy"]])
        scale = np.abs(ref_terms).max()
        assert np.abs(terms[q].cpu().numpy() - ref_terms).max() <= LOSS_TOL * scale, (q, terms[q], ref_terms)
        assert abs(float(loss[q]) - ref) <= LOSS_TOL * scale
        for n, t in zip(GRAD_NAMES, grads):
            e = rel_l2(t[q].cpu().numpy().astype(np.float64) / float(gl[q]), gref[n])
            assert e < GRAD_TOL, (q, n, e)


@pytest.mark.parametrize("nprob,Bx,By,T,D,two_pairs", [(20, 24, 40, 5, 64, True), (33, 64, 64, 4, 96, True),
                                                       (16, 8, 16, 3, 32, False)])
def test_cost_many_problems_abi(nprob, Bx, By, T, D, two_pairs):
    """kccot_cost_fwd with many problems per call (the per-problem finalize kernel: one and two martingale pairs,
    rectangular blocks): sampled problems against single-problem calls (tile finalize kernel) and against fp64
    s * (|x_i - y_j|^2 + sum_pairs sum_t h_i,t (M_j,t+1 - M_j,t))  (gan_utils.py:14-17, :34-38, :59-66)."""
    from kccotgan_b200 import _lib, functional as F
    lib = _lib.load()
    J, s = 5, 1.0 / 9.0
    K = T * D
    g = torch.Generator().manual_seed(7 * nprob + Bx)
    x = torch.rand((nprob, Bx, T, D), generator=g)
    y = torch.rand((nprob, By, T, D), generator=g)
    h1, h2 = [torch.sigmoid(torch.randn((nprob, Bx, T, J), generator=g)) for _ in range(2)]     # row-indexed
    M1, M2 = [torch.sigmoid(torch.randn((nprob, By, T, J), generator=g)) for _ in range(2)]     # column-indexed
    dx, dy, dh1, dM1, dh2, dM2 = [t.cuda().contiguous() for t in (x, y, h1, M1, h2, M2)]
    p, st = F._ptr, F._stream(dx.device)
    C = torch.full((nprob, Bx, By), float("nan"), device="cuda")
    ws = torch.empty(lib.kccot_cost_workspace_bytes(nprob, Bx, By, K), dtype=torch.uint8, device="cuda")
    _lib.call("kccot_cost_fwd", p(dx), p(dy), nprob, Bx, By, K, p(dh1), p(dM1), p(dh2) if two_pairs else None,
              p(dM2) if two_pairs else None, T, J, s, p(C), p(ws), ws.numel(), 0, st)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(C).all())
    for q in (0, nprob // 2, nprob - 1):
        Cq = torch.empty((Bx, By), device="cuda")
        wsq = torch.empty(lib.kccot_cost_workspace_bytes(1, Bx, By, K), dtype=torch.uint8, device="cuda")
        _lib.call("kccot_cost_fwd", p(dx[q]), p(dy[q]), 1, Bx, By, K, p(dh1[q]), p(dM1[q]), p(dh2[q]) if two_pairs else None,
                  p(dM2[q]) if two_pairs else None, T, J, s, p(Cq), p(wsq), wsq.numel(), 0, st)
        torch.cuda.synchronize()
        assert maxrel(C[q].cpu(), Cq.cpu()) < COST_TOL
        xx, yy = x[q].numpy().astype(np.float64).reshape(Bx, -1), y[q].numpy().astype(np.float64).reshape(By, -1)
        ref = (xx * xx).sum(1)[:, None] + (yy * yy).sum(1)[None, :] - 2.0 * xx @ yy.T
        for hh, MM in ((h1, M1), (h2, M2))[: 2 if two_pairs else 1]:
            hq, Mq = hh[q].numpy().astype(np.float64), MM[q].numpy().astype(np.float64)
            ref = ref + np.einsum("itk,jtk->ij", hq[:, :-1], Mq[:, 1:] - Mq[:, :-1])
        assert maxrel(C[q].cpu(), s * ref) < COST_TOL


# ---------------------------------------------------------------------------------------------
# Sinkhorn kernels in isolation against the fp64 oracle on the same (fp32-rounded) cost
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,eps,L", [(64, 1.0, 100), (32, 0.8, 100), (17, 0.3, 40), (64, 1.0, 250), (96, 1.0, 60),
                                     (200, 0.7, 30), (96, 2.0, 300), (64, 1.0, 600), (8, 0.5, 100), (98, 1.0, 40),
                                     (302, 0.7, 25), (98, 2.0, 300)])
def test_sinkhorn_kernels_vs_oracle(B, eps, L):
    from kccotgan_b200 import _lib
    from kccotgan_b200.functional import SinkhornFn
    from oracle import closed_form as cf
    rng = np.random.default_rng(B + L)
    C = (900.0 + 4.0 * rng.standard_normal((2, B, B))).astype(np.float32)
    C[1] = np.abs(C[1] - 900.0) * 3.0                     # a small-valued problem next to a large-valued one
    Ct = torch.from_numpy(C).cuda().requires_grad_(True)
    n0 = _lib.load().kccot_launch_count()
    cost, nits = SinkhornFn.apply(Ct, eps, L, 100, 1e-2, False)
    if B > 64 and B % 4:
        # the persistent kernel needs B % 4 == 0, so these shapes must take the streamed fallback: at least two
        # launches per iteration and problem
        assert _lib.load().kccot_launch_count() - n0 >= 2 * L * len(C)
    w = torch.tensor([1.0, -2.0], device="cuda")
    gC, = torch.autograd.grad((cost * w).sum(), Ct)
    for n in range(2):
        ref, uh, vh, rn = cf.sinkhorn_forward(C[n].astype(np.float64), eps, L, Lmin=100, thresh=1e-2)
        assert int(nits[n]) == rn, (int(nits[n]), rn)
        assert abs(float(cost[n]) - ref) <= LOSS_TOL * abs(ref), (float(cost[n]), ref)
        Cb = cf.sinkhorn_backward(C[n].astype(np.float64), eps, uh, vh, rn, gbar=float(w[n]))
        e = rel_l2(gC[n].cpu().numpy(), Cb)
        print(B, eps, L, n, "nits", rn, "cost rel", abs(float(cost[n]) - ref) / abs(ref), "Cbar rel-L2", e)
        assert e < GRAD_TOL


@pytest.mark.parametrize("B,L,kind", [(64, 100, "diag"), (40, 100, "diag"), (64, 400, "diag"), (64, 100, "slow"),
                                      (24, 100, "slow"), (64, 10, "diag")])
def test_sinkhorn_history_fixed_point(B, L, kind):
    """The forward kernel stops iterating once the fp32 scalings repeat bit for bit and fills the rest of
    the history with copies (sinkhorn_small.cu): every saved row must still equal the potentials the
    reference's L iterations produce.  "diag" reaches the fixed point after one iteration (the xx / yy
    problems of the mixed loss), "slow" after some tens of iterations."""
    from kccotgan_b200 import _lib, functional as F
    from oracle import closed_form as cf
    rng = np.random.default_rng(7 * B + L)
    if kind == "diag":
        C = (500.0 * (1.0 - np.eye(B)) + rng.random((B, B))).astype(np.float32)
    else:
        C = (1350.0 + 30.0 * rng.random((B, B))).astype(np.float32)
    Ct = torch.from_numpy(C[None]).cuda()
    uh = torch.full((1, L + 1, B), float("nan"), device="cuda")
    vh = torch.full((1, L + 1, B), float("nan"), device="cuda")
    nits = torch.zeros(1, dtype=torch.int32, device="cuda")
    cost = torch.zeros(1, device="cuda")
    ws = torch.empty(_lib.load().kccot_sinkhorn_workspace_bytes(1, B, L), dtype=torch.uint8, device="cuda")
    _lib.call("kccot_sinkhorn_fwd", F._ptr(Ct), 1, B, 1.0, L, 100, 1e-2, 0, F._ptr(uh), F._ptr(vh), F._ptr(nits),
              F._ptr(cost), F._ptr(ws), ws.numel(), F._stream(Ct.device))
    C64 = C.astype(np.float64)
    ref, ruh, rvh, rn = cf.sinkhorn_forward(C64 - C64.min(), 1.0, L, Lmin=100, thresh=1e-2)
    assert int(nits[0]) == rn
    ln2 = np.log(2.0)                                   # saved potentials are in log2 units of the shifted cost
    gu, gv = uh[0, : rn + 1].cpu().numpy() * ln2, vh[0, : rn + 1].cpu().numpy() * ln2
    assert np.isfinite(gu).all() and np.isfinite(gv).all()
    scale = max(np.abs(ruh).max(), np.abs(rvh).max(), 1.0)
    eu, ev = np.abs(gu - ruh[: rn + 1]).max() / scale, np.abs(gv - rvh[: rn + 1]).max() / scale
    print(kind, B, L, "nits", rn, "history err", eu, ev)
    assert eu < 1e-5 and ev < 1e-5
    assert abs(float(cost[0]) - (ref + C64.min())) <= LOSS_TOL * abs(ref + C64.min())


@pytest.mark.parametrize("B,eps,L", [(24, 0.02, 30), (64, 0.05, 120), (40, 0.01, 10)])
def test_sinkhorn_guard_path(B, eps, L):
    """Ill-scaled problems (spread/eps in the hundreds) leave the fp32 range of the scaling form: the
    kernels must roll back to the log-domain updates and still match the oracle."""
    from kccotgan_b200.functional import SinkhornFn
    from oracle import closed_form as cf
    rng = np.random.default_rng(B + L)
    C = (900.0 + 4.0 * rng.standard_normal((2, B, B))).astype(np.float32)
    C[1] = np.abs(C[1] - 900.0) * 3.0
    Ct = torch.from_numpy(C).cuda().requires_grad_(True)
    cost, nits = SinkhornFn.apply(Ct, eps, L, 100, 1e-2, False)
    gC, = torch.autograd.grad(cost.sum(), Ct)
    assert torch.isfinite(cost).all() and torch.isfinite(gC).all()
    for n in range(2):
        ref, uh, vh, rn = cf.sinkhorn_forward(C[n].astype(np.float64), eps, L, Lmin=100, thresh=1e-2)
        Cb = cf.sinkhorn_backward(C[n].astype(np.float64), eps, uh, vh, rn)
        e = rel_l2(gC[n].cpu().numpy(), Cb)
        print("guard", B, eps, L, n, "nits", int(nits[n]), rn, "cost rel", abs(float(cost[n]) - ref) / abs(ref), "Cbar", e)
        assert int(nits[n]) == rn
        assert abs(float(cost[n]) - ref) <= LOSS_TOL * abs(ref)
        assert e < 2e-3          # eps this small makes the plan a near-permutation: ill-conditioned gradient


@pytest.mark.parametrize("B,na,nb,D", [(32, 20, 12, 150.0), (64, 40, 24, 200.0)])
def test_sinkhorn_guard_trips_late(B, na, nb, D):
    """Two unbalanced clusters behind a cost barrier: the potentials drift by ~0.5 per iteration and the scaling
    form leaves its fp32 range only around iteration 115 — after the tight loop (Lmin = 100 < L = 150), in the
    loop whose roll-back used to be decided through an unsynchronised flag (ADVICE r1, sinkhorn_small.cu)."""
    from kccotgan_b200.functional import SinkhornFn
    from oracle import closed_form as cf
    rng = np.random.default_rng(0)
    C = np.full((B, B), D)
    C[:na, :nb] = 0.0
    C[na:, nb:] = 0.0
    C = (C + rng.random((B, B))).astype(np.float32)
    L = 150
    for rep in range(3):                                  # a race shows up as a hang or as run-to-run differences
        Ct = torch.from_numpy(C[None]).cuda().requires_grad_(True)
        cost, nits = SinkhornFn.apply(Ct, 1.0, L, 100, 1e-2, False)
        gC, = torch.autograd.grad(cost.sum(), Ct)
        ref, uh, vh, rn = cf.sinkhorn_forward(C.astype(np.float64), 1.0, L, Lmin=100, thresh=1e-2)
        Cb = cf.sinkhorn_backward(C.astype(np.float64), 1.0, uh, vh, rn)
        e = rel_l2(gC[0].cpu().numpy(), Cb)
        print("late guard", B, "nits", int(nits[0]), rn, "cost", float(cost[0]), ref, "Cbar", e)
        assert int(nits[0]) == rn
        assert abs(float(cost[0]) - ref) <= LOSS_TOL * max(abs(ref), 1.0)
        assert e < 2e-3


# ---------------------------------------------------------------------------------------------
# smoothing
# ---------------------------------------------------------------------------------------------
def test_smoothing_golden():
    from kccotgan_b200.data_utils import KernelSmoothing
    g = load_golden("smoothing.npz")
    ks = KernelSmoothing(temporal_kernel_size=6, spatial_kernel_size=6)
    for sig in (5.0, 1.7):
        assert rel_l2(ks.gaussian_kernel1d(3, sig).cpu().numpy(), g[f"kernel1d_sigma{sig}"]) < 1e-6
        assert rel_l2(ks.gaussian_kernel3d(3, sig).cpu().numpy(), g[f"kernel3d_sigma{sig}"]) < 1e-6
    assert ks.annealing_sigma(5.0, 1000) == float(g["annealing_sigma_5_1000"])
    with pytest.raises(ValueError):
        ks.spatial_convolution(torch.rand(2, 8, 5, 8, 3, device="cuda"), 5.0)
    for tag in ("nc3", "nc1", "tie"):
        for mode, fn in (("1d", ks.temporal_convolution), ("3d", ks.gaussian_convolution3D)):
            for sig in (5.0, 1.7):
                x = dev(g[f"x_{tag}"], grad=True)
                out = fn(x, sig)
                gx, = torch.autograd.grad(out, x, dev(g[f"gout_{tag}"]))
                eo = rel_l2(out.detach().cpu().numpy(), g[f"{mode}_{tag}_sigma{sig}"])
                eg = rel_l2(gx.cpu().numpy(), g[f"{mode}_{tag}_sigma{sig}_grad"])
                assert float(out.max()) == 1.0
                assert eo < 1e-5 and eg < GRAD_TOL, (tag, mode, sig, eo, eg)


def test_smoothing_full_frame():
    """64x64x3 frames (cfg 3 shape at reduced batch) against the fp64 oracle."""
    from kccotgan_b200.data_utils import KernelSmoothing
    from oracle import closed_form as cf
    ks = KernelSmoothing(6, 6)
    torch.manual_seed(3)
    x = torch.rand(3, 64, 12, 64, 3)
    go = torch.randn(3, 64, 12, 64, 3)
    for mode, fn, cfn in (("1d", ks.temporal_convolution, cf.temporal_convolution),
                          ("3d", ks.gaussian_convolution3D, cf.gaussian_convolution3D)):
        xl = x.cuda().requires_grad_(True)
        out = fn(xl, 5.0)
        gx, = torch.autograd.grad(out, xl, go.cuda())
        ro, rg = cfn(x.numpy(), 5.0, grad_out=go.numpy())
        assert rel_l2(out.detach().cpu().numpy(), ro) < 1e-5, mode
        assert rel_l2(gx.cpu().numpy(), rg) < GRAD_TOL, mode


@pytest.mark.parametrize("shape", [(2, 9, 7, 10, 1), (3, 16, 5, 12, 3), (1, 4, 4, 5, 2), (2, 64, 20, 64, 1),
                                   (2, 12, 9, 7, 4), (5, 8, 64, 6, 1)])
def test_smoothing_shapes(shape):
    """Shapes that exercise both filter kernels (register-window columns, shared-memory tiles), the scalar
    (inner % 4 != 0) and vector paths, single-channel frames and the axis-length limits."""
    from kccotgan_b200.data_utils import KernelSmoothing
    from oracle import closed_form as cf
    ks = KernelSmoothing(6, 6)
    g = torch.Generator().manual_seed(sum(shape))
    x = torch.rand(shape, generator=g)
    go = torch.randn(shape, generator=g)
    for mode, fn, cfn in (("1d", ks.temporal_convolution, cf.temporal_convolution),
                          ("3d", ks.gaussian_convolution3D, cf.gaussian_convolution3D)):
        xl = x.cuda().requires_grad_(True)
        out = fn(xl, 2.5)
        gx, = torch.autograd.grad(out, xl, go.cuda())
        ro, rg = cfn(x.numpy(), 2.5, grad_out=go.numpy())
        assert float(out.max()) == 1.0
        assert rel_l2(out.detach().cpu().numpy(), ro) < 1e-5, (mode, shape)
        assert rel_l2(gx.cpu().numpy(), rg) < GRAD_TOL, (mode, shape)


@pytest.mark.parametrize("tk,sk,shape", [
    (8, 8, (2, 12, 10, 12, 3)),       # the class's own default spatial size 8 -> radius 4 (VERDICT r1: raised)
    (6, 8, (2, 16, 7, 16, 1)),        # KernelSmoothing() defaults: temporal radius 3, spatial radius 4
    (2, 3, (3, 6, 5, 6, 2)),          # radius 1
    (12, 12, (1, 16, 14, 16, 1)),     # radius 6
    (6, 6, (1, 96, 8, 80, 1)),        # axes longer than 64
    (6, 6, (1, 8, 200, 4, 1)),        # a long temporal axis
])
def test_smoothing_radius_and_axis_range(tk, sk, shape):
    from kccotgan_b200.data_utils import KernelSmoothing
    from oracle import closed_form as cf
    ks = KernelSmoothing(temporal_kernel_size=tk, spatial_kernel_size=sk)
    g = torch.Generator().manual_seed(tk * 100 + sk)
    x = torch.rand(shape, generator=g)
    go = torch.randn(shape, generator=g)
    for mode, fn, cfn, r in (("1d", ks.temporal_convolution, cf.temporal_convolution, tk // 2),
                             ("3d", ks.gaussian_convolution3D, cf.gaussian_convolution3D, sk // 2)):
        xl = x.cuda().requires_grad_(True)
        out = fn(xl, 2.0)
        gx, = torch.autograd.grad(out, xl, go.cuda())
        ro, rg = cfn(x.numpy(), 2.0, radius=r, grad_out=go.numpy())
        assert float(out.max()) == 1.0
        assert rel_l2(out.detach().cpu().numpy(), ro) < 1e-5, (mode, shape)
        assert rel_l2(gx.cpu().numpy(), rg) < GRAD_TOL, (mode, shape)
    with pytest.raises((ValueError, RuntimeError)):
        KernelSmoothing(30, 30).temporal_convolution(torch.rand(1, 4, 40, 4, 1, device="cuda"), 2.0)     # radius 15


def test_smoothing_annealed_sigma_is_graph_capturable():
    """The filter weights are kernel arguments: a smoothing call with a never-seen sigma copies nothing to the
    device, so it can sit inside a CUDA-graph capture (ADVICE r1: the dense filter matrix was rebuilt on the host
    and copied from pageable memory for every new sigma)."""
    from kccotgan_b200.data_utils import KernelSmoothing
    from oracle import closed_form as cf
    ks = KernelSmoothing(6, 6)
    x = torch.rand(2, 8, 6, 8, 1)
    xd = x.cuda()
    sig = ks.annealing_sigma(5.0, 12345)
    ks.temporal_convolution(xd, 4.0)                     # warm-up with a different sigma
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        out = ks.temporal_convolution(xd, sig)
    gr.replay()
    torch.cuda.synchronize()
    ro = cf.temporal_convolution(x.numpy(), sig)
    assert rel_l2(out.cpu().numpy(), ro) < 1e-5


@pytest.mark.parametrize("kernel", ["none", "1d", "3d"])
def test_training_step_closures(kernel):
    """kernel_train.py:219-292 with stub networks (kccotgan_b200.train_step): the loss the generator step
    sees equals the fp64 oracle on the same tensors, both steps update exactly the parameters the
    reference updates, and everything stays finite over a few iterations."""
    from kccotgan_b200 import gan_utils
    from kccotgan_b200.data_utils import KernelSmoothing
    from kccotgan_b200.train_step import StubDiscriminator, StubGenerator, make_training_steps
    from oracle import closed_form as cf
    B, H, T, ctx, W, C = 8, 16, 6, 2, 16, 3
    torch.manual_seed(5)
    gen = StubGenerator(T - ctx, C).cuda()
    dh, dm = StubDiscriminator(H, W, C).cuda(), StubDiscriminator(H, W, C).cuda()
    disc_step, gen_step = make_training_steps(gen, dh, dm, B, kernel_choice=kernel, gen_lr=1e-2, disc_lr=1e-2)
    x = torch.rand(B, H, T, W, C, device="cuda")
    real_in, real_pred = x[:, :, :ctx], x[:, :, ctx:]
    # the loss of the first generator forward against the oracle on the very same tensors
    with torch.no_grad():
        z = torch.randn(B, gen.z_dim, device="cuda")
        fake = torch.cat((real_in, gen(real_in, z)), dim=2)
        real = x
        ks = KernelSmoothing(6, 6)
        if kernel == "1d":
            real, fake = ks.temporal_convolution(real, 5.0), ks.temporal_convolution(fake, 5.0)
        elif kernel == "3d":
            real, fake = ks.gaussian_convolution3D(real, 5.0), ks.gaussian_convolution3D(fake, 5.0)
        hf, hr, mr, mf = dh(fake), dh(real), dm(real), dm(fake)
        loss = gan_utils.compute_sinkhorn_loss(real, fake, 1 / 15, 0.8, 100, hf, mr, hr, mf, video=True)
        a = [t.cpu().numpy().astype(np.float64) for t in (real, fake, hf, mr, hr, mf)]
        ref, _, det = cf.compute_sinkhorn_loss(a[0], a[1], 1 / 15, 0.8, 100, a[2], a[3], a[4], a[5], grad=True)
        scale = max(abs(det["loss_xy"]), abs(det["loss_xx"]), abs(det["loss_yy"]))
        assert abs(float(loss) - ref) <= LOSS_TOL * scale
    before = [p.detach().clone() for m in (gen, dh, dm) for p in m.parameters()]
    ngen = len(list(gen.parameters()))
    pm = disc_step(real_in, real_pred, 5.0)
    after_d = [p.detach().clone() for m in (gen, dh, dm) for p in m.parameters()]
    assert all(torch.equal(b, a) for b, a in zip(before[:ngen], after_d[:ngen]))          # generator untouched (:252-255)
    assert all(not torch.equal(b, a) for b, a in zip(before[ngen:], after_d[ngen:]))      # both discriminators moved
    loss = gen_step(real_in, real_pred, 5.0)
    after_g = [p.detach().clone() for m in (gen, dh, dm) for p in m.parameters()]
    assert all(not torch.equal(b, a) for b, a in zip(after_d[:ngen], after_g[:ngen]))     # generator moved (:289-291)
    assert all(torch.equal(b, a) for b, a in zip(after_d[ngen:], after_g[ngen:]))
    for _ in range(3):
        pm, loss = disc_step(real_in, real_pred, 5.0), gen_step(real_in, real_pred, 5.0)
    assert np.isfinite(float(pm)) and np.isfinite(float(loss))                             # kernel_train.py:323


def test_c_abi_from_plain_c(gu, tmp_path):
    """examples/mixed_loss_demo.c drives the C ABI with nothing but the CUDA runtime: its loss, terms and
    gradient checksums must equal the Python host path on the same (LCG-generated) inputs, and the loss the
    fp64 oracle."""
    import subprocess
    from test_abi import _build_c_demo
    from oracle import closed_form as cf
    exe = _build_c_demo(tmp_path)
    B, T, H, W, C, J = 16, 6, 8, 8, 3, 8
    r = subprocess.run([exe, str(B), str(T), str(H), str(W), str(C)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = dict()
    for line in r.stdout.splitlines():
        w = line.split()
        if w[0] == "loss":
            out.update(loss=float(w[1]), xy=float(w[3]), xx=float(w[5]), yy=float(w[7]))
        elif w[0] == "grad":
            out["g_" + w[1]] = float(w[2])
    state = 12345
    def draw(n, lo, hi):
        nonlocal state
        a = np.empty(n, dtype=np.float32)
        for i in range(n):
            state = (state * 1664525 + 1013904223) & 0xFFFFFFFF
            a[i] = np.float32(lo) + (np.float32(hi) - np.float32(lo)) * (np.float32(state >> 8) * np.float32(1.0 / 16777216.0))
        return a
    K = T * H * W * C
    real = draw(B * K, 0, 1).reshape(B, T, H * W * C)
    fake = draw(B * K, 0, 1).reshape(B, T, H * W * C)
    hm = [draw(B * T * J, 0.1, 0.9).reshape(B, T, J) for _ in range(4)]
    leaves = [torch.from_numpy(a).cuda().requires_grad_(True) for a in (real, fake, *hm)]
    loss = gu.compute_sinkhorn_loss(leaves[0], leaves[1], 1 / 15, 0.8, 100, *leaves[2:], video=False)
    grads = torch.autograd.grad(loss, leaves)
    assert abs(out["loss"] - float(loss)) <= 1e-6 * max(abs(out["xy"]), 1.0)
    for n, g in zip(GRAD_NAMES, grads):
        flat = g.detach().cpu().numpy().reshape(-1).astype(np.float64)
        ck = float((flat * (1 + np.arange(flat.size) % 7)).sum())
        assert abs(out["g_" + n] - ck) <= 1e-5 * (np.abs(flat).sum() * 7 + 1e-12), (n, out["g_" + n], ck)
    ref, _, det = cf.compute_sinkhorn_loss(real, fake, 1 / 15, 0.8, 100, *hm, grad=True)
    scale = max(abs(det["loss_xy"]), abs(det["loss_xx"]), abs(det["loss_yy"]))
    assert abs(out["loss"] - ref) <= LOSS_TOL * scale and abs(out["xy"] - det["loss_xy"]) <= LOSS_TOL * scale


def test_errors_raise(gu):
    x = torch.rand(8, 4, 16, device="cuda")
    with pytest.raises(ValueError):
        gu.cost_xy(x.cpu(), x, 0.1)
    with pytest.raises(ValueError):
        gu.cost_xy(x.double(), x.double(), 0.1)
    with pytest.raises(ValueError):
        gu.cost_xy(x, torch.rand(8, 4, 12, device="cuda"), 0.1)
    with pytest.raises(ValueError):
        gu.compute_sinkhorn_loss(x, x, 0.1, 1.0, 100, x, x, x, x, video=True)


# ---------------------------------------------------------------------------------------------
# batched Python entry point (BASELINE config 4's shape) and its CUDA-graph replay
# ---------------------------------------------------------------------------------------------
def test_batched_entry_point_cfg4_shape(gu):
    """256 x (B=64, T=10, 32x32x1): a sample of the problems against the fp64 oracle, and eps = 0.8 by keyword."""
    from oracle import closed_form as cf
    s = 1.0 / 15.0
    P, B, T, H, W, C = 256, 64, 10, 32, 32, 1
    g = torch.Generator().manual_seed(4)
    real = torch.rand((P, B, H, T, W, C), generator=g)
    fake = torch.rand((P, B, H, T, W, C), generator=g)
    hm = [torch.sigmoid(torch.randn((P, B, T, 8), generator=g)) for _ in range(4)]
    lv = [t.cuda().requires_grad_(True) for t in (real, fake, *hm)]
    loss = gu.compute_sinkhorn_loss_batched(lv[0], lv[1], s, *lv[2:])
    w = torch.linspace(0.5, 1.5, P).cuda()
    grads = torch.autograd.grad((loss * w).sum(), lv[1:])
    for q in (0, 117, 255):
        a = [t[q].numpy().astype(np.float64) for t in (real, fake, *hm)]
        ref, gref, det = cf.compute_sinkhorn_loss(a[0], a[1], s, 0.8, 100, *a[2:], grad=True)
        scale = max(abs(det["loss_xy"]), abs(det["loss_xx"]), abs(det["loss_yy"]))
        assert abs(float(loss[q]) - ref) <= LOSS_TOL * scale, (q, float(loss[q]), ref)
        for n, gt in zip(GRAD_NAMES[1:], grads):
            e = rel_l2(gt[q].cpu().numpy().astype(np.float64) / float(w[q]), gref[n])
            assert e < GRAD_TOL, (q, n, e)


def test_batched_graph_replay_many_problems():
    """Queued CUDA-graph replays of a many-problem chain (150+ problems: every kernel runs in several waves) must keep
    making progress.  They used to hang about once in a few hundred evaluations: the gradient GEMM dealt its boxes
    round-robin to converter warps that did not own a ring slot, and a parity wait passed a pass early when TMA
    loads completed out of order (csrc/grad_tcgen05.cu, converter branch).  Runs in a child process under a timeout."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "scripts", "batched_graph_probe2.py"), "160", "2", "1", "400"],
                       capture_output=True, text=True, timeout=180, cwd=root)
    assert r.returncode == 0 and "400 alternating replays ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_evaluation_lanes_match_serial_replays():
    """Independent evaluations replayed on separate streams (EvaluationLanes) leave exactly the results of serial
    replays: every evaluator owns its buffers, nothing is shared between lanes."""
    from kccotgan_b200.graphed import EvaluationLanes, GraphedSinkhornLoss
    from kccotgan_b200.synthetic import INPUT_ORDER, make_inputs
    dev = torch.device("cuda", 0)
    evs = []
    for i in range(4):
        inp = make_inputs(B=32, T=6, H=16, W=16, C=3, J=8, ctx=2, kind="uniform" if i % 2 else "video", seed=40 + i,
                          device=dev)
        evs.append(GraphedSinkhornLoss(*[inp[k] for k in INPUT_ORDER], 1.0 / 15.0, adopt=True))
    ref = []
    for ev in evs:
        ev.step()
        torch.cuda.synchronize()
        ref.append((float(ev.loss), {k: v.clone() for k, v in ev.grads.items()}))
        with torch.no_grad():
            ev.loss.detach().zero_()
            for v in ev.grads.values():
                v.detach().zero_()
    lanes = EvaluationLanes(evs, n_lanes=3)
    assert len(lanes) == 4 and len(lanes.streams) == 3
    lanes.fork()
    for rep in range(5):
        for j in range(len(lanes)):
            lanes.submit(j)
    lanes.join()
    torch.cuda.synchronize()
    for ev, (l, g) in zip(evs, ref):
        assert float(ev.loss) == l
        for k in g:
            assert torch.equal(ev.grads[k], g[k]), k
    with pytest.raises(ValueError):
        EvaluationLanes([])


@pytest.mark.parametrize("B,T,ctx,H,W,C", [(64, 10, 3, 8, 32, 3), (32, 20, 10, 4, 32, 1), (16, 6, 2, 4, 8, 3)])
def test_shared_context_hint(gu, B, T, ctx, H, W, C):
    """compute_sinkhorn_loss_shared_context (SURVEY §8 f3; kernel_train.py:225-226): on videos whose first ctx frames
    are shared, the loss is bit-identical to the plain call, the gradient of the predicted frames and of h / M is
    bit-identical, the gradient of fake's context frames is zero; fake's context frames are never read (poisoned
    with NaN here).  The last shape (W*C = 24, not a multiple of 32) exercises the fallback."""
    dev = torch.device("cuda", 0)
    s = 1.0 / 15.0
    inp = make_inputs(B=B, T=T, H=H, W=W, C=C, J=8, ctx=ctx, kind="video", seed=11, device=dev)
    lv = [inp[k].clone().requires_grad_(k != "real") for k in INPUT_ORDER]
    loss0 = gu.compute_sinkhorn_loss(lv[0], lv[1], s, 0.8, 100, *lv[2:], video=True)
    g0 = torch.autograd.grad(loss0, lv[1:])
    usable = (W * C) % 32 == 0
    fake2 = inp["fake"].clone()
    if usable:
        fake2[:, :, :ctx] = float("nan")            # must not be read
    lv2 = [inp["real"].clone(), fake2.requires_grad_(True)] + [inp[k].clone().requires_grad_(True) for k in INPUT_ORDER[2:]]
    loss1, terms1 = gu.compute_sinkhorn_loss_shared_context(lv2[0], lv2[1], s, *lv2[2:], ctx_frames=ctx)
    g1 = torch.autograd.grad(loss1, lv2[1:])
    torch.cuda.synchronize()
    assert float(loss1) == float(loss0)
    assert torch.equal(g1[0][:, :, ctx:], g0[0][:, :, ctx:])
    assert float(g1[0][:, :, :ctx].abs().max()) == 0.0
    assert float(g0[0][:, :, :ctx].abs().max()) > 0.0
    for a, b in zip(g1[1:], g0[1:]):
        assert torch.equal(a, b)
    with pytest.raises(ValueError):
        gu.compute_sinkhorn_loss_shared_context(lv2[0], lv2[1], s, *lv2[2:], ctx_frames=T)


@pytest.mark.parametrize("kernel", ["none", "1d"])
def test_graphed_training_iteration_matches_eager(kernel):
    """GraphedTrainingIteration replays exactly what the eager step closures do: same noise stream (default CUDA
    generator, same seed), same parameters after three iterations, same loss / pM."""
    from kccotgan_b200.train_step import GraphedTrainingIteration, StubDiscriminator, StubGenerator, make_training_steps
    B, H, T, ctx, W, C = 8, 16, 6, 2, 16, 3
    x = [torch.rand(B, H, T, W, C, device="cuda", generator=torch.Generator(device="cuda").manual_seed(70 + i)) for i in range(3)]

    def build():
        torch.manual_seed(9)
        gen = StubGenerator(T - ctx, C).cuda()
        dh, dm = StubDiscriminator(H, W, C).cuda(), StubDiscriminator(H, W, C).cuda()
        return gen, dh, dm

    # eager run with the capturable optimisers (the default generator drives the noise in both runs)
    gen, dh, dm = build()
    disc_step, gen_step = make_training_steps(gen, dh, dm, B, kernel_choice=kernel, gen_lr=1e-2, disc_lr=1e-2, capturable=True)
    warm = 2
    torch.manual_seed(123)
    for _ in range(warm):                                       # mirrors the warm-up iterations of the graphed object
        disc_step(x[0][:, :, :ctx], x[0][:, :, ctx:], 5.0)
        gen_step(x[0][:, :, :ctx], x[0][:, :, ctx:], 5.0)
    outs = []
    for i in range(3):
        pm = disc_step(x[i][:, :, :ctx], x[i][:, :, ctx:], 5.0)
        loss = gen_step(x[i][:, :, :ctx], x[i][:, :, ctx:], 5.0)
        outs.append((float(loss), float(pm)))
    ref_params = [p.detach().clone() for m in (gen, dh, dm) for p in m.parameters()]

    gen2, dh2, dm2 = build()
    torch.manual_seed(123)
    it = GraphedTrainingIteration(gen2, dh2, dm2, x[0][:, :, :ctx], x[0][:, :, ctx:], sigma=5.0, warmup=warm,
                                  kernel_choice=kernel, gen_lr=1e-2, disc_lr=1e-2)
    # (the capture pass itself does not execute and does not advance the generator's offset beyond what replays use)
    for i in range(3):
        it.real_in.copy_(x[i][:, :, :ctx])
        it.real_pred.copy_(x[i][:, :, ctx:])
        loss, pm = it.step()
        torch.cuda.synchronize()
        assert np.isfinite(float(loss)) and np.isfinite(float(pm))
        assert abs(float(loss) - outs[i][0]) <= 1e-4 * max(1.0, abs(outs[i][0])), (i, float(loss), outs[i])
        assert abs(float(pm) - outs[i][1]) <= 1e-4 * max(1.0, abs(outs[i][1])), (i, float(pm), outs[i])
    if kernel == "none":      # (with the 1d kernel the smoothing adjoint sums with atomics: Adam turns last-bit gradient
        for a, b in zip(ref_params, [p for m in (gen2, dh2, dm2) for p in m.parameters()]):      # noise into +-lr steps)
            assert torch.allclose(a, b, rtol=2e-3, atol=2e-5)
