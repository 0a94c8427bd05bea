"""T0/T1: the oracle (closed_form.py, port_torch.py) against the golden vectors produced by the
reference's own source (oracle/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from conftest import golden_inputs, load_golden, rel_l2
from oracle import closed_form as cf
from oracle import port_torch as pt
from kccotgan_b200.synthetic import INPUT_ORDER, GRAD_NAMES

TOL = 1e-11   # fp64 restatement vs fp64 execution of the reference source


@pytest.fixture(scope="module")
def small():
    return load_golden("gan_utils_small.npz")


def test_cost_functions(small):
    g = small
    s = float(g["scaling_coef"])
    assert rel_l2(cf.cost_xy(g["x"], g["y"], s), g["cost_xy"]) < TOL
    assert rel_l2(cf.modified_cost(g["x"], g["y"], g["hy"], g["Mx"], s), g["modified_cost"]) < TOL
    assert rel_l2(cf.bi_causal_modified_cost(g["x"], g["y"], g["hy"], g["Mx"], g["hx"], g["My"], s),
                  g["bi_causal_modified_cost"]) < TOL
    assert rel_l2(cf.compute_N(g["Mx"][:, :, 0]), g["compute_N"]) < TOL


def test_crossed_indices_quirk(small):
    """SURVEY §0.5: h is indexed by the row sample, Delta M by the column sample."""
    g = small
    s = float(g["scaling_coef"])
    hm = g["modified_cost"] - g["cost_xy"]
    Ht, dM = cf.martingale_operands(g["hy"], g["Mx"])
    assert rel_l2(s * Ht @ dM.T, hm) < 1e-9
    assert rel_l2(s * dM @ Ht.T, hm) > 1e-2      # the "paper" orientation is NOT what runs


@pytest.mark.parametrize("tag,kw", [("default", {}), ("eps0p8", dict(epsilon=0.8)),
                                    ("eps0p3_L20", dict(epsilon=0.3, L=20)), ("L130", dict(L=130)),
                                    ("eps5_L400", dict(epsilon=5.0, L=400))])
def test_compute_sinkhorn(small, tag, kw):
    g = small
    s = float(g["scaling_coef"])
    c, o = cf.compute_sinkhorn(g["x"], g["y"], g["hy"], g["Mx"], s, grad=True, **kw)
    assert abs(c - float(g[f"compute_sinkhorn_{tag}"])) <= TOL * abs(c)
    for n in ("x", "y", "hy", "Mx"):
        assert rel_l2(o[n], g[f"compute_sinkhorn_{tag}_grad_{n}"]) < 1e-9, n


def test_early_exit_only_beyond_100(small):
    """SURVEY §0.7: Lmin=100 is hard-coded; only L>100 can stop early."""
    g = small
    s = float(g["scaling_coef"])
    C = cf.modified_cost(g["x"], g["y"], g["hy"], g["Mx"], s)
    assert cf.sinkhorn_forward(C, 1.0, 100)[3] == 100
    assert cf.sinkhorn_forward(C, 5.0, 400)[3] == 100      # converged long before -> exits at Lmin
    assert cf.sinkhorn_forward(C, 1.0, 37)[3] == 37


def test_bicausal(small):
    g = small
    s = float(g["scaling_coef"])
    c, o = cf.compute_sinkhorn(g["x"], g["y"], g["hy"], g["Mx"], s, g["hx"], g["My"], epsilon=0.5, L=50,
                               bi_causal=True, grad=True)
    assert abs(c - float(g["compute_sinkhorn_bicausal"])) <= TOL * abs(c)
    for n in ("x", "y", "hy", "Mx", "hx", "My"):
        assert rel_l2(o[n], g[f"compute_sinkhorn_bicausal_grad_{n}"]) < 1e-9, n


@pytest.mark.parametrize("tag,kw", [("default", {}), ("eps0p5_L40_Lmin5", dict(epsilon=0.5, L=40, Lmin=5)),
                                    ("eps2_L200_Lmin10", dict(epsilon=2.0, L=200, Lmin=10))])
def test_benchmark_sinkhorn(small, tag, kw):
    g = small
    c = cf.benchmark_sinkhorn(g["x"], g["y"], float(g["scaling_coef"]), **kw)
    assert abs(c - float(g[f"benchmark_sinkhorn_{tag}"])) <= TOL * abs(c)


def test_eps_l_arguments_ignored(small):
    """SURVEY §0.4: compute_sinkhorn_loss's eps/L land in hx/My and are ignored."""
    g = small
    s = float(g["scaling_coef"])
    a = cf.compute_sinkhorn_loss(g["x"], g["y"], s, 0.8, 100, g["hy"], g["Mx"], g["hx"], g["My"], video=False)
    b = cf.compute_sinkhorn_loss(g["x"], g["y"], s, 5.0, 7, g["hy"], g["Mx"], g["hx"], g["My"], video=False)
    assert a == b
    assert abs(a - float(g["loss_novideo"])) <= 1e-10 * max(1.0, abs(a))


def test_pm(small):
    g = small
    for tag, M in (("a", g["Mx"]), ("b", g["My"])):
        pm, gm = cf.martingale_regularization(M, 1.3, float(g["scaling_coef"]), grad=True)
        assert abs(pm - float(g[f"pm_{tag}"])) <= TOL * abs(pm)
        assert rel_l2(gm, g[f"pm_{tag}_grad"]) < 1e-9


@pytest.mark.parametrize("cfg", ["cfg1", "cfg2", "cfg3"])
@pytest.mark.parametrize("kind", ["uniform", "video"])
def test_mixed_loss_reduced(cfg, kind):
    g = load_golden(f"loss_{cfg}_reduced_{kind}.npz")
    s = float(g["scaling_coef"])
    inp = golden_inputs(g)          # the golden inputs are exactly what synthetic.make_inputs re-draws from the seed
    args = [inp[k].numpy() for k in INPUT_ORDER]
    loss, grads, det = cf.compute_sinkhorn_loss(args[0], args[1], s, 0.8, 100, *args[2:], grad=True)
    scale = max(abs(float(g[k])) for k in ("loss_xy", "loss_xx", "loss_yy"))
    assert abs(loss - float(g["loss"])) <= 1e-10 * scale
    for k in ("loss_xy", "loss_xx", "loss_yy"):
        assert abs(det[k] - float(g[k])) <= 1e-10 * scale
    for k in ("C_xy", "C_xx", "C_yy"):
        assert rel_l2(det[k], g[k]) < TOL
    for n in GRAD_NAMES:
        assert rel_l2(grads[n], g["grad_" + n]) < 1e-8, n


def test_port_matches_golden_fp64_and_fp32():
    """The torch port of the reference formulation (the CPU baseline that bench.py times)."""
    g = load_golden("loss_cfg2_reduced_uniform.npz")
    s = float(g["scaling_coef"])
    inp = golden_inputs(g)
    t64 = [inp[k].double() for k in INPUT_ORDER]
    loss, grads = pt.mixed_loss_fwd_bwd(t64[0], t64[1], s, *t64[2:])
    assert abs(float(loss) - float(g["loss"])) < 1e-9 * abs(float(g["loss_xy"]))
    for n in GRAD_NAMES[1:]:
        assert rel_l2(grads[n].numpy(), g["grad_" + n]) < 1e-8, n
    t32 = [inp[k].float() for k in INPUT_ORDER]
    loss32, grads32 = pt.mixed_loss_fwd_bwd(t32[0], t32[1], s, *t32[2:])
    # fp32 run of the same formulation reproduces the reference's own fp32 numbers closely; of the video gradient
    # the golden keeps a fixed sample of elements
    assert abs(float(loss32) - float(g["loss_f32"])) < 2e-4 * abs(float(g["loss_xy"]))
    idx = g["grad_f32_sample_index"]
    for n in GRAD_NAMES[1:]:
        got = grads32[n].numpy()
        ref = g.get("grad_" + n + "_f32")
        if ref is None:
            got, ref = got.reshape(-1)[idx], g["grad_" + n + "_f32_sample"]
        assert rel_l2(got, ref) < 2e-3, n


def test_smoothing_golden():
    g = load_golden("smoothing.npz")
    assert bool(g["2d_raises"])
    for sig in (5.0, 1.7):
        assert rel_l2(cf.gaussian_kernel1d(3, sig), g[f"kernel1d_sigma{sig}"]) < 1e-7   # fp32 weights upstream
        assert rel_l2(cf.gaussian_kernel3d(3, sig), g[f"kernel3d_sigma{sig}"]) < 1e-6
    assert abs(cf.annealing_sigma(5.0, 1000) - float(g["annealing_sigma_5_1000"])) < 1e-12
    assert abs(cf.annealing_sigma(5.0, 12345) - float(g["annealing_sigma_5_12345"])) < 1e-12
    for tag in ("nc3", "nc1", "tie"):
        for mode, fn in (("1d", cf.temporal_convolution), ("3d", cf.gaussian_convolution3D)):
            for sig in (5.0, 1.7):
                out, gx = fn(g[f"x_{tag}"], sig, grad_out=g[f"gout_{tag}"])
                assert rel_l2(out, g[f"{mode}_{tag}_sigma{sig}"]) < 1e-10, (tag, mode, sig)
                assert rel_l2(gx, g[f"{mode}_{tag}_sigma{sig}_grad"]) < 1e-9, (tag, mode, sig)


def test_smoothing_output_max_is_one():
    x = np.random.default_rng(0).random((2, 8, 6, 8, 3))
    assert cf.temporal_convolution(x, 5.0).max() == 1.0
    assert cf.gaussian_convolution3D(x, 5.0).max() == 1.0
    with pytest.raises(ValueError):
        cf.temporal_convolution(x[:, :, :3], 5.0)        # REFLECT needs T > radius


def test_translation_invariance_and_zero_diagonal():
    rng = np.random.default_rng(3)
    x = rng.random((5, 4, 7))
    y = rng.random((5, 4, 7))
    c = rng.random((1, 4, 7))
    assert np.allclose(cf.cost_xy(x, y, 0.1), cf.cost_xy(x + c, y + c, 0.1), rtol=1e-12, atol=1e-12)
    assert np.all(np.diag(cf.cost_xy(x, x, 0.1)) == 0.0)


def test_plan_column_marginals():
    """After the v-update the column marginals of pi are exact (1/B)."""
    rng = np.random.default_rng(4)
    C = rng.random((9, 9)) * 3
    _, uh, vh, n = cf.sinkhorn_forward(C, 0.7, 25)
    pi = np.exp((uh[n][:, None] + vh[n][None, :] - C) / 0.7)
    assert np.allclose(pi.sum(axis=0), 1.0 / 9, rtol=1e-12)


def test_backward_finite_difference():
    rng = np.random.default_rng(5)
    C = rng.random((6, 6)) * 2
    eps, L = 0.6, 15
    _, uh, vh, n = cf.sinkhorn_forward(C, eps, L)
    Cb = cf.sinkhorn_backward(C, eps, uh, vh, n)
    num = np.zeros_like(C)
    for i in range(6):
        for j in range(6):
            d = np.zeros_like(C)
            d[i, j] = 1e-6
            num[i, j] = (cf.sinkhorn_forward(C + d, eps, L)[0] - cf.sinkhorn_forward(C - d, eps, L)[0]) / 2e-6
    assert rel_l2(Cb, num) < 1e-7
