"""bf16 entry points of the row-sharded cost, host side and compiled footprint (no GPU needed).

The entry points reject null pointers, a bad row range and video or gradient pointers that are not 16-byte aligned
with KCCOT_EINVAL before any CUDA call.  The bf16 pre-pass kernels do not spill; the bf16 instantiation of the
adjoint GEMM spills no more than the fp32 one it shares its main loop with.  Footprints are read from the built
library as in test_footprint.py.
"""
import ctypes

import pytest

from kccotgan_b200 import _lib
from test_footprint import _dump, _one, _res_usage


@pytest.fixture(scope="module")
def lib():
    from kccotgan_b200 import build
    build.build()
    return _lib.load()


@pytest.mark.parametrize("kernel", ["colsum_part_bf16_kernel", "split_bf16_kernel"])
def test_bf16_prepass_kernels_do_not_spill(lib, kernel):
    reg, stack, local = _one(_res_usage(), kernel)
    assert stack == 0 and local == 0, f"{kernel}: stack {stack}, local {local} bytes (spills)"
    assert kernel in _dump("-symbols")


def test_bf16_gemm_spills_no_more_than_fp32(lib):
    usage = _res_usage()
    f32 = [v for n, v in usage.items() if "gemm_f16x3_pair_kernelIfE" in n]
    b16 = [v for n, v in usage.items() if "gemm_f16x3_pair_kernelItE" in n]
    assert len(f32) == 1 and len(b16) == 1, sorted(n for n in usage if "gemm_f16x3" in n)
    assert b16[0][0] <= f32[0][0] and b16[0][1] <= f32[0][1] and b16[0][2] <= f32[0][2], (b16, f32)


P = ctypes.c_void_p
GOOD = P(0x10000)                  # never dereferenced: every call below fails its argument check first
BAD = P(0x10002)


def _fwd(lib, real=GOOD, fake=GOOD, h=GOOD, row0=0, Brows=8, B=8, K=128, ws=GOOD):
    return lib.kccot_shard_cost_fwd_bf16(real, fake, B, K, row0, Brows, h, GOOD, GOOD, GOOD, 2, 1, 1.0, GOOD, ws,
                                         1 << 20, None)


def _bwd(lib, g=GOOD, cbar=GOOD, row0=0, Brows=8, B=8, K=128):
    return lib.kccot_shard_cost_bwd_bf16(cbar, GOOD, GOOD, B, K, row0, Brows, GOOD, GOOD, GOOD, GOOD, 2, 1, 1.0, g,
                                         GOOD, GOOD, GOOD, GOOD, GOOD, 1 << 20, None)


def test_null_pointers_are_rejected(lib):
    for kw in ({"real": None}, {"fake": None}, {"h": None}, {"ws": None}):
        assert _fwd(lib, **kw) == _lib.EINVAL and "null" in _lib.last_error(), kw
    assert _bwd(lib, cbar=None) == _lib.EINVAL and "null" in _lib.last_error()


def test_misaligned_pointers_are_rejected(lib):
    assert _fwd(lib, real=BAD) == _lib.EINVAL and "aligned" in _lib.last_error()
    assert _fwd(lib, fake=BAD) == _lib.EINVAL and "aligned" in _lib.last_error()
    assert _bwd(lib, g=BAD) == _lib.EINVAL and "aligned" in _lib.last_error()


@pytest.mark.parametrize("row0, Brows", [(-1, 4), (0, 0), (6, 4), (8, 1)])
def test_bad_row_range_is_rejected(lib, row0, Brows):
    assert _fwd(lib, row0=row0, Brows=Brows) == _lib.EINVAL and "row range" in _lib.last_error()
    assert _bwd(lib, row0=row0, Brows=Brows) == _lib.EINVAL and "row range" in _lib.last_error()

