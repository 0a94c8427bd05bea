"""Generate tests/golden/*.npz by EXECUTING THE REFERENCE'S OWN SOURCE (container only).

TEST INFRASTRUCTURE.  Run:  python -m oracle.make_golden
Everything stored is an output of `/root/reference/gan_utils.py` / `data_utils.py:478-586`
running on torch CPU through `oracle/tf_shim`, in fp64 unless the key ends in `_f32`, with
gradients from autograd through the reference's unrolled graph.  Inputs are fp32-representable
(drawn in fp32, then widened), so the CUDA path sees bit-identical inputs.
"""
import hashlib
import os
import sys
import warnings

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kccotgan_b200.synthetic import make_inputs, INPUT_ORDER, GRAD_NAMES  # noqa: E402
from oracle import ref_exec  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
S = 1.0 / 15.0


def _np(t):
    return t.detach().numpy().copy()


def _loss_case(g, inp, dtype):
    leaves = [inp[k].to(dtype).clone().requires_grad_(True) for k in INPUT_ORDER]
    r, f, hf, mr, hr, mf = leaves
    loss = g.compute_sinkhorn_loss(r, f, S, 0.8, 100, hf, mr, hr, mf, video=True)
    grads = torch.autograd.grad(loss, leaves)
    with torch.no_grad():
        rt = r.permute(0, 2, 1, 3, 4).reshape(r.shape[0], r.shape[2], -1)
        ft = f.permute(0, 2, 1, 3, 4).reshape(f.shape[0], f.shape[2], -1)
        terms = dict(loss_xy=g.compute_sinkhorn(rt, ft, hf, mr, S), loss_xx=g.compute_sinkhorn(rt, rt, hr, mr, S),
                     loss_yy=g.compute_sinkhorn(ft, ft, hf, mf, S))
        C = dict(C_xy=g.modified_cost(rt, ft, hf, mr, S), C_xx=g.modified_cost(rt, rt, hr, mr, S),
                 C_yy=g.modified_cost(ft, ft, hf, mf, S))
    return loss, grads, terms, C


F32_SAMPLE = 4096


def reduced_record(d, seed, J):
    """What a reduced-size case stores, so that each file stays below 1 MB: instead of the inputs their SHA-256
    digests (`sha256_<input>`; the tests re-draw the inputs with synthetic.make_inputs from `seed` and check them),
    every fp64 result in full, and of the fp32 gradients of the two videos the same fixed seeded sample of elements
    (`grad_f_real_f32_sample`, `grad_f_fake_f32_sample` at the flat indices `grad_f32_sample_index`).  `d` holds
    the inputs and every result in full."""
    out = {k: v for k, v in d.items() if k not in INPUT_ORDER}
    out.update({"sha256_" + k: np.str_(hashlib.sha256(np.ascontiguousarray(d[k]).tobytes()).hexdigest())
                for k in INPUT_ORDER})
    out.update(seed=seed, J=J)
    idx = np.sort(np.random.default_rng(0).choice(d["real"].size, F32_SAMPLE, replace=False)).astype(np.int32)
    out["grad_f32_sample_index"] = idx
    for n in ("f_real", "f_fake"):
        out[f"grad_{n}_f32_sample"] = out.pop(f"grad_{n}_f32").reshape(-1)[idx]
    return out


def gen_loss_reduced(g):
    """BASELINE configs 1-3 at reduced frame size (full B, T, J); see reduced_record for what is stored."""
    cases = {"cfg1": dict(B=32, T=20, ctx=10, H=8, W=8, C=1), "cfg2": dict(B=64, T=10, ctx=3, H=4, W=4, C=3),
             "cfg3": dict(B=64, T=12, ctx=2, H=4, W=4, C=3)}
    for name, c in cases.items():
        for kind in ("uniform", "video"):
            inp = make_inputs(J=8, kind=kind, seed=1, **c)
            loss, grads, terms, C = _loss_case(g, inp, torch.float64)
            loss32, grads32, _, _ = _loss_case(g, inp, torch.float32)
            d = {k: _np(inp[k]) for k in INPUT_ORDER}
            d.update(loss=float(loss), loss_f32=float(loss32), scaling_coef=S, kind=kind, **c)
            d.update({k: float(v) for k, v in terms.items()})
            d.update({k: _np(v) for k, v in C.items()})
            d.update({"grad_" + n: _np(gr) for n, gr in zip(GRAD_NAMES, grads)})
            d.update({"grad_" + n + "_f32": _np(gr) for n, gr in zip(GRAD_NAMES, grads32)})
            np.savez_compressed(os.path.join(OUT, f"loss_{name}_reduced_{kind}.npz"), **reduced_record(d, seed=1, J=8))
            print(name, kind, float(loss), flush=True)


def gen_loss_full(g):
    """Full-size configs: inputs are re-drawn from the seed by the test; only outputs stored
    (the video gradient as norm + strided sample + a random projection)."""
    from kccotgan_b200.synthetic import CONFIGS
    for name, kinds in (("cfg1_mmnist", ("uniform", "video")), ("cfg2_mazes", ("uniform",))):
        c = {k: v for k, v in CONFIGS[name].items() if k != "nprob"}
        for kind in kinds:
            inp = make_inputs(J=8, kind=kind, seed=1, **c)
            loss, grads, terms, C = _loss_case(g, inp, torch.float64)
            d = dict(loss=float(loss), scaling_coef=S, kind=kind, seed=1, J=8, **c)
            d.update({k: float(v) for k, v in terms.items()})
            d.update({k: _np(v) for k, v in C.items()})
            for n, gr in zip(GRAD_NAMES, grads):
                a = _np(gr)
                if a.size > 100000:
                    flat = a.reshape(-1)
                    probe = np.random.default_rng(7).standard_normal(flat.size)
                    d["grad_" + n + "_norm"] = float(np.linalg.norm(flat))
                    d["grad_" + n + "_stride"] = 997
                    d["grad_" + n + "_sample"] = flat[::997].copy()
                    d["grad_" + n + "_proj"] = float(flat @ probe)
                else:
                    d["grad_" + n] = a
            np.savez_compressed(os.path.join(OUT, f"loss_{name}_full_{kind}.npz"), **d)
            print(name, kind, float(loss), flush=True)


def _store_grads(d, grads, prefix="grad_"):
    for n, gr in zip(GRAD_NAMES, grads):
        a = _np(gr)
        if a.size > 100000:
            flat = a.reshape(-1)
            probe = np.random.default_rng(7).standard_normal(flat.size)
            d[prefix + n + "_norm"] = float(np.linalg.norm(flat))
            d[prefix + n + "_stride"] = 997
            d[prefix + n + "_sample"] = flat[::997].copy()
            d[prefix + n + "_proj"] = float(flat @ probe)
        else:
            d[prefix + n] = a


def gen_loss_full_cfg3(g):
    """BASELINE config 3 at full size (B=64, 2+10 frames of 64x64x3), uniform inputs: the loss alone, and the
    chain kernel_train.py:270-288 runs with `--kernel 1d`: temporal smoothing (sigma = 5) of real and fake, then
    the loss on the smoothed tensors, gradients back to the UNSMOOTHED inputs."""
    from kccotgan_b200.synthetic import CONFIGS
    KS = ref_exec.load_kernel_smoothing()
    ks = KS(temporal_kernel_size=6, spatial_kernel_size=6)
    c = {k: v for k, v in CONFIGS["cfg3_bair"].items() if k != "nprob"}
    inp = make_inputs(J=8, kind="uniform", seed=1, **c)
    loss, grads, terms, C = _loss_case(g, inp, torch.float64)
    d = dict(loss=float(loss), scaling_coef=S, kind="uniform", seed=1, J=8, **c)
    d.update({k: float(v) for k, v in terms.items()})
    d.update({k: _np(v) for k, v in C.items()})
    _store_grads(d, grads)
    del grads, C
    # smoothing -> loss
    leaves = [inp[k].to(torch.float64).clone().requires_grad_(True) for k in INPUT_ORDER]
    r, f, hf, mr, hr, mf = leaves
    rs, fs = ks.temporal_convolution(r, 5.0), ks.temporal_convolution(f, 5.0)
    loss_s = g.compute_sinkhorn_loss(rs, fs, S, 0.8, 100, hf, mr, hr, mf, video=True)
    grads_s = torch.autograd.grad(loss_s, leaves)
    d["smooth1d_loss"] = float(loss_s)
    d["smooth1d_sigma"] = 5.0
    with torch.no_grad():
        rt = rs.permute(0, 2, 1, 3, 4).reshape(rs.shape[0], rs.shape[2], -1)
        ft = fs.permute(0, 2, 1, 3, 4).reshape(fs.shape[0], fs.shape[2], -1)
        d["smooth1d_loss_xy"] = float(g.compute_sinkhorn(rt, ft, hf, mr, S))
        d["smooth1d_loss_xx"] = float(g.compute_sinkhorn(rt, rt, hr, mr, S))
        d["smooth1d_loss_yy"] = float(g.compute_sinkhorn(ft, ft, hf, mf, S))
        flat = _np(fs).reshape(-1)
        d["smooth1d_fake_sample"] = flat[::997].copy()
        d["smooth1d_fake_norm"] = float(np.linalg.norm(flat))
    _store_grads(d, grads_s, prefix="smooth1d_grad_")
    np.savez_compressed(os.path.join(OUT, "loss_cfg3_bair_full_uniform.npz"), **d)
    print("cfg3 full", float(loss), float(loss_s), flush=True)


def gen_gan_utils_small(g):
    """Every gan_utils function (rows a1-a8 of SURVEY §8) on one tiny case, plus the quirk KATs."""
    torch.manual_seed(11)
    B, T, D, J = 6, 5, 12, 3
    f32 = lambda *s: torch.rand(*s, dtype=torch.float32)  # noqa: E731
    x, y = f32(B, T, D), f32(B, T, D)
    hy, Mx, hx, My = (torch.sigmoid(torch.randn(B, T, J, dtype=torch.float32)) for _ in range(4))
    d = dict(x=_np(x), y=_np(y), hy=_np(hy), Mx=_np(Mx), hx=_np(hx), My=_np(My), scaling_coef=S)
    X, Y, HY, MX, HX, MY = (t.double() for t in (x, y, hy, Mx, hx, My))
    d["cost_xy"] = _np(g.cost_xy(X, Y, S))
    d["modified_cost"] = _np(g.modified_cost(X, Y, HY, MX, S))
    d["bi_causal_modified_cost"] = _np(g.bi_causal_modified_cost(X, Y, HY, MX, HX, MY, S))
    d["compute_N"] = _np(g.compute_N(MX[:, :, 0]))
    for tag, kw in {"default": {}, "eps0p8": dict(epsilon=0.8), "eps0p3_L20": dict(epsilon=0.3, L=20),
                    "L130": dict(L=130), "eps5_L400": dict(epsilon=5.0, L=400)}.items():
        lv = [t.clone().requires_grad_(True) for t in (X, Y, HY, MX)]
        c = g.compute_sinkhorn(lv[0], lv[1], lv[2], lv[3], S, **kw)
        gr = torch.autograd.grad(c, lv)
        d[f"compute_sinkhorn_{tag}"] = float(c)
        for n, a in zip(("x", "y", "hy", "Mx"), gr):
            d[f"compute_sinkhorn_{tag}_grad_{n}"] = _np(a)
    lv = [t.clone().requires_grad_(True) for t in (X, Y, HY, MX, HX, MY)]
    c = g.compute_sinkhorn(lv[0], lv[1], lv[2], lv[3], S, lv[4], lv[5], epsilon=0.5, L=50, bi_causal=True)
    gr = torch.autograd.grad(c, lv)
    d["compute_sinkhorn_bicausal"] = float(c)
    for n, a in zip(("x", "y", "hy", "Mx", "hx", "My"), gr):
        d[f"compute_sinkhorn_bicausal_grad_{n}"] = _np(a)
    for tag, kw in {"default": {}, "eps0p5_L40_Lmin5": dict(epsilon=0.5, L=40, Lmin=5),
                    "eps2_L200_Lmin10": dict(epsilon=2.0, L=200, Lmin=10)}.items():
        lv = [t.clone().requires_grad_(True) for t in (X, Y)]
        c = g.benchmark_sinkhorn(lv[0], lv[1], S, **kw)
        gr = torch.autograd.grad(c, lv)
        d[f"benchmark_sinkhorn_{tag}"] = float(c)
        d[f"benchmark_sinkhorn_{tag}_grad_x"] = _np(gr[0])
        d[f"benchmark_sinkhorn_{tag}_grad_y"] = _np(gr[1])
    # quirk KAT (SURVEY §0.4): eps/L arguments of compute_sinkhorn_loss are ignored
    a = g.compute_sinkhorn_loss(X, Y, S, 0.8, 100, HY, MX, HX, MY, video=False)
    b = g.compute_sinkhorn_loss(X, Y, S, 5.0, 7, HY, MX, HX, MY, video=False)
    assert float(a) == float(b)
    d["loss_novideo"] = float(a)
    # p_M
    for tag, M in {"a": MX, "b": MY}.items():
        Ml = M.clone().requires_grad_(True)
        pm = g.scale_invariante_martingale_regularization(Ml, 1.3, S)
        gm, = torch.autograd.grad(pm, Ml)
        d[f"pm_{tag}"] = float(pm)
        d[f"pm_{tag}_grad"] = _np(gm)
    np.savez_compressed(os.path.join(OUT, "gan_utils_small.npz"), **d)
    print("gan_utils_small ok", flush=True)


def gen_smoothing():
    KS = ref_exec.load_kernel_smoothing()
    ks = KS(temporal_kernel_size=6, spatial_kernel_size=6)
    torch.manual_seed(5)
    d = {}
    for sig in (5.0, 1.7):
        d[f"kernel1d_sigma{sig}"] = _np(ks.gaussian_kernel1d(3, sig).double())
        d[f"kernel3d_sigma{sig}"] = _np(ks.gaussian_kernel3d(3, sig).double())
    d["annealing_sigma_5_1000"] = ks.annealing_sigma(5.0, 1000)
    d["annealing_sigma_5_12345"] = ks.annealing_sigma(5.0, 12345)
    cases = {"nc3": (2, 9, 6, 8, 3), "nc1": (3, 8, 7, 10, 1), "tie": (2, 8, 5, 8, 1)}
    for tag, shp in cases.items():
        x = torch.rand(*shp, dtype=torch.float32)
        if tag == "tie":
            x[1] = x[0]                      # two samples identical -> the global max is attained twice
        go = torch.randn(*shp, dtype=torch.float32)
        d[f"x_{tag}"], d[f"gout_{tag}"] = _np(x), _np(go)
        for mode, fn in (("1d", ks.temporal_convolution), ("3d", ks.gaussian_convolution3D)):
            for sig in (5.0, 1.7):
                xl = x.double().requires_grad_(True)
                out = fn(xl, sig)
                gx, = torch.autograd.grad(out, xl, go.double())
                d[f"{mode}_{tag}_sigma{sig}"] = _np(out)
                d[f"{mode}_{tag}_sigma{sig}_grad"] = _np(gx)
    try:
        ks.spatial_convolution(torch.rand(2, 8, 5, 8, 3).double(), 5.0)
        d["2d_raises"] = False
    except Exception:
        d["2d_raises"] = True
    np.savez_compressed(os.path.join(OUT, "smoothing.npz"), **d)
    print("smoothing ok", flush=True)


def main():
    warnings.simplefilter("ignore")
    os.makedirs(OUT, exist_ok=True)
    torch.set_default_dtype(torch.float64)   # the reference's tf.float32 -> fp64 (see tf_shim)
    g = ref_exec.load_gan_utils()
    if "--only-cfg3" in sys.argv:
        gen_loss_full_cfg3(g)
        return
    gen_gan_utils_small(g)
    gen_smoothing()
    gen_loss_reduced(g)
    if "--no-full" not in sys.argv:
        gen_loss_full(g)
        gen_loss_full_cfg3(g)


if __name__ == "__main__":
    main()
