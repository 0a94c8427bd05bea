"""The C-ABI library builds, loads, and exports every symbol include/kccot.h declares; host-side
argument validation.  CPU only (no compute calls)."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from kccotgan_b200 import build, _lib
    build.build()
    return _lib.load()


def test_header_symbols_exported(lib):
    from kccotgan_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "kccot.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(kccot_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in kccot.h but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)


def test_version_and_no_cpu_fallback(lib):
    from kccotgan_b200 import _lib
    assert lib.kccot_version() == 203
    if not torch.cuda.is_available():
        assert lib.kccot_device_check() != 0
        assert "no CUDA device" in _lib.last_error()


def test_header_constants_match_the_python_table():
    """KCCOT_VERSION and KCCOT_SHARD_FLAGS_PER_RANK of include/kccot.h against kccotgan_b200/_lib.py."""
    import os
    import re
    from kccotgan_b200 import _lib
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "kccot.h")).read()
    assert int(re.search(r"#define\s+KCCOT_SHARD_FLAGS_PER_RANK\s+(\d+)", hdr).group(1)) == _lib.SHARD_FLAGS_PER_RANK
    assert int(re.search(r"#define\s+KCCOT_VERSION\s+(\d+)", hdr).group(1)) == _lib.load().kccot_version()
    # the shared-context entry points reject a hint whose length is not below its period (no CUDA call involved)
    rc = _lib.load().kccot_mixed_loss_fwd_ctx(None, None, 1, 8, 64, None, None, None, None, 2, 1, 1.0, 1.0, 1, None, None, None,
                                              None, 0, 0, None, 32, 32)
    assert rc == _lib.EINVAL and "shared-context" in _lib.last_error()


def test_workspace_queries(lib):
    assert lib.kccot_mixed_cost_workspace_bytes(1, 64, 122880) > 0
    assert lib.kccot_cost_workspace_bytes(1, 64, 64, 1000) > 0
    assert lib.kccot_sinkhorn_workspace_bytes(3, 64, 100) >= 256
    assert lib.kccot_sinkhorn_workspace_bytes(1, 512, 100) > 512 * 4 * 4
    assert lib.kccot_smooth_workspace_bytes(3, 2, 8, 8, 8, 1) >= 2 * 2 * 8 * 8 * 8 * 4
    assert lib.kccot_cost_workspace_bytes(0, 64, 64, 1000) == 0


def test_argument_errors_are_value_errors(lib):
    from kccotgan_b200 import _lib
    with pytest.raises(ValueError):
        _lib.call("kccot_cost_fwd", None, None, 1, 8, 8, 64, None, None, None, None, 0, 0, 0.1, None, None, 0, 0, None)
    with pytest.raises(ValueError):
        _lib.call("kccot_smooth_fwd", 2, None, 1, 8, 8, 8, 1, None, 3, None, 3, None, None, None, 0, None)
    assert "2d" in _lib.last_error()


def test_python_surface_matches_reference_signatures():
    """Same names / positional orders / defaults as gan_utils.py and KernelSmoothing."""
    import inspect
    from kccotgan_b200 import gan_utils as g
    from kccotgan_b200.data_utils import KernelSmoothing
    sig = lambda f: str(inspect.signature(f))  # noqa: E731
    assert sig(g.cost_xy) == "(x, y, scaling_coef)"
    assert sig(g.modified_cost) == "(x, y, h, M, scaling_coef)"
    assert sig(g.bi_causal_modified_cost) == "(x, y, hy, Mx, hx, My, scaling_coef)"
    assert sig(g.benchmark_sinkhorn) == "(x, y, scaling_coef, epsilon=1.0, L=10, Lmin=10)"
    assert sig(g.compute_sinkhorn) == "(x, y, hy, Mx, scaling_coef, hx=None, My=None, epsilon=1.0, L=100, bi_causal=False)"
    assert sig(g.compute_N) == "(M)"
    assert sig(g.scale_invariante_martingale_regularization) == "(M, reg_lam, scaling_coef)"
    assert sig(g.compute_sinkhorn_loss) == ("(f_real, f_fake, scaling_coef, sinkhorn_eps, sinkhorn_l, h_fake, m_real, "
                                            "h_real, m_fake, video=True)")
    assert sig(KernelSmoothing.__init__) == "(self, temporal_kernel_size=6, spatial_kernel_size=8)"
    assert sig(KernelSmoothing.annealing_sigma) == "(self, init_sigma, step, decay_steps=500, decay_rate=0.975)"
    ks = KernelSmoothing(6, 6)
    assert ks.temporal_radius == 3 and ks.spatial_radius == 3
    assert ks.annealing_sigma(5.0, 1000) == 5.0 * 0.975 ** 2


def test_cpu_tensors_rejected():
    from kccotgan_b200 import gan_utils as g
    x = torch.rand(4, 3, 8)
    with pytest.raises(ValueError, match="CUDA"):
        g.cost_xy(x, x, 0.1)
    with pytest.raises(ValueError):
        g.compute_sinkhorn_loss(x, x, 0.1, 1.0, 100, x, x, x, x, video=False)


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under kccotgan_b200/ may reference it."""
    pkg = os.path.join(ROOT, "kccotgan_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), fn
            assert "oracle." not in src and "/oracle" not in src, fn


def test_smoothing_weights_match_oracle():
    """The host side only produces the 2r+1 weights (the REFLECT band is formed inside the kernels): same numbers
    as the reference's gaussian_kernel1d for every radius the library takes, default constructor included."""
    import numpy as np
    from kccotgan_b200.data_utils import KernelSmoothing
    from oracle import closed_form as cf
    ks = KernelSmoothing()                       # reference defaults: temporal 6 -> radius 3, spatial 8 -> radius 4
    assert (ks.temporal_radius, ks.spatial_radius) == (3, 4)
    for r in range(1, 7):
        for sigma in (0.7, 1.7, 5.0):
            w = ks._weights(r, sigma)
            assert w.shape == (2 * r + 1,) and w.dtype == np.float32
            assert np.allclose(w, cf.gaussian_kernel1d(r, sigma), atol=1e-7)
            assert abs(float(w.sum()) - 1.0) < 1e-6


def test_header_is_plain_c(tmp_path):
    """include/kccot.h is the drop-in boundary: it must compile as C (no C++ or torch types) and every
    prototype must match the ctypes table used by the Python host (count and pointer-vs-scalar kinds)."""
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = os.path.join(root, "include", "kccot.h")
    src = tmp_path / "t.c"
    src.write_text('#include "kccot.h"\nint (*probe)(void) = kccot_version;\nint main(void) { return probe == 0; }\n')
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.dirname(hdr), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    from kccotgan_b200 import _lib
    text = re.sub(r"/\*.*?\*/", "", open(hdr).read(), flags=re.S)
    protos = re.findall(r"\b(kccot_\w+)\s*\(([^;{]*?)\)\s*;", text)
    assert protos
    for name, args in protos:
        assert name in _lib.SIGNATURES, name
        args = [a.strip() for a in args.split(",") if a.strip() and a.strip() != "void"]
        _, ctypes_args = _lib.SIGNATURES[name]
        assert len(args) == len(ctypes_args), (name, len(args), len(ctypes_args))
        for a, ct in zip(args, ctypes_args):
            is_ptr = "*" in a
            assert is_ptr == (ct is _lib._P), (name, a, ct)


def _build_c_demo(tmp_path):
    import subprocess
    root = ROOT
    exe = str(tmp_path / "mixed_loss_demo")
    libdir = os.path.join(root, "kccotgan_b200")
    cmd = ["gcc", "-O2", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(root, "include"), "-I", "/usr/local/cuda/include",
           os.path.join(root, "examples", "mixed_loss_demo.c"), "-L", libdir, "-lkccot", "-L", "/usr/local/cuda/lib64", "-lcudart",
           "-Wl,-rpath," + libdir, "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_c_demo_links_and_fails_loudly_without_gpu(lib, tmp_path):
    """examples/mixed_loss_demo.c (plain C, no PyTorch) links against libkccot.so; without a device it must
    exit with an error instead of computing anything on the host."""
    import subprocess
    exe = _build_c_demo(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("covered by the GPU test")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 2 and "no CUDA device" in r.stderr
