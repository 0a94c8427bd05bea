"""Batched martingale penalty, host side and compiled footprint (no GPU needed).

kccot_pm_batched_fwd / _bwd compute nprob independent penalties in one call.  Every argument error (those of
kccot_pm_fwd / _bwd, plus a problem count outside 1..65535) is reported as KCCOT_EINVAL before any CUDA call, the header
declares both entries as the ctypes table does, neither batched kernel spills, and the Python function rejects a CPU
tensor before anything reaches the device.
"""
import ctypes
import os
import re

import pytest
import torch

from kccotgan_b200 import _lib
from test_footprint import _res_usage

P = ctypes.c_void_p
GOOD = P(0x10000)                  # never dereferenced: every call below fails its argument check first
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from kccotgan_b200 import build
    build.build()
    return _lib.load()


def _fwd(lib, M=GOOD, nprob=3, B=64, T=10, J=8, pm=GOOD, stats=GOOD):
    return lib.kccot_pm_batched_fwd(M, nprob, B, T, J, 1.0, 0.1, pm, stats, None)


def _bwd(lib, M=GOOD, nprob=3, B=64, T=10, J=8, stats=GOOD, gpm=GOOD, gM=GOOD):
    return lib.kccot_pm_batched_bwd(M, nprob, B, T, J, 1.0, 0.1, stats, gpm, gM, None)


ENTRIES = [_fwd, _bwd]
POINTERS = {_fwd: ("M", "pm", "stats"), _bwd: ("M", "stats", "gpm", "gM")}


@pytest.fixture(autouse=True)
def _no_launch(request):
    """every call here fails before any CUDA call: the library's launch counter does not move"""
    if "lib" not in request.fixturenames:
        yield
        return
    lib = request.getfixturevalue("lib")
    before = lib.kccot_launch_count()
    yield
    assert lib.kccot_launch_count() == before


@pytest.mark.parametrize("call", ENTRIES)
def test_null_pointers(lib, call):
    for name in POINTERS[call]:
        assert call(lib, **{name: None}) == _lib.EINVAL and "null" in _lib.last_error(), name


@pytest.mark.parametrize("call", ENTRIES)
def test_problem_count(lib, call):
    for nprob in (0, -1, 65536):
        assert call(lib, nprob=nprob) == _lib.EINVAL and "nprob" in _lib.last_error(), nprob


@pytest.mark.parametrize("call", ENTRIES)
def test_sizes(lib, call):
    for kw in (dict(B=0), dict(B=-3), dict(T=1), dict(T=0), dict(J=0), dict(J=-1)):
        assert call(lib, **kw) == _lib.EINVAL and "bad sizes" in _lib.last_error(), kw


def test_shared_memory_cap(lib):
    """the forward holds two [T*J] rows in shared memory, up to 48 KB, as kccot_pm_fwd does"""
    for T, J in ((2, 6136), (6000, 3), (1537, 4)):
        assert (2 * T * J + 2 * J + 32) * 4 > 48 * 1024
        assert _fwd(lib, T=T, J=J) == _lib.EINVAL and "too large" in _lib.last_error(), (T, J)
        assert lib.kccot_pm_fwd(GOOD, 64, T, J, 1.0, 0.1, GOOD, GOOD, None) == _lib.EINVAL


def test_header_declares_the_ctypes_table():
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "kccot.h")).read(), flags=re.S)
    protos = dict(re.findall(r"\b(kccot_pm_batched_\w+)\s*\(([^;{]*?)\)\s*;", text))
    assert set(protos) == {"kccot_pm_batched_fwd", "kccot_pm_batched_bwd"}
    for name, args in protos.items():
        args = [a.strip() for a in args.split(",")]
        _, ctypes_args = _lib.SIGNATURES[name]
        assert len(args) == len(ctypes_args), name
        assert [("*" in a) for a in args] == [ct is _lib._P for ct in ctypes_args], name
        assert args[1] == "int nprob", name                 # the problem count follows M, as in the batched loss


def test_batched_pm_kernels_do_not_spill(lib):
    found = {n: v for n, v in _res_usage().items() if re.search(r"\d(pm_batched_fwd_kernel|pm_batched_bwd_kernel)E", n)}
    assert len(found) == 2, sorted(found)
    spills = {n: v for n, v in found.items() if v[1] or v[2]}
    assert not spills, spills


def test_python_rejects_cpu_tensors():
    from kccotgan_b200 import gan_utils
    for dtype in (torch.float32, torch.bfloat16, torch.float64):
        with pytest.raises(ValueError, match="CUDA"):
            gan_utils.scale_invariante_martingale_regularization_batched(torch.rand(3, 8, 5, 2).to(dtype), 1.0, 0.1)
    with pytest.raises(ValueError, match="torch.Tensor"):
        gan_utils.scale_invariante_martingale_regularization_batched([[[[1.0]]]], 1.0, 0.1)
