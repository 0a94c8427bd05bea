"""bf16 entry points of the mixed loss, host side and compiled footprint (no GPU needed).

The bf16 gradient kernel keeps the fp32 kernel's half-SM footprint (two CTAs per SM: registers x threads <= 32 768)
and neither bf16 kernel spills; the footprint is read from the built library as in test_footprint.py.  The entry
points reject KCCOT_FLAG_ACCUMULATE and misaligned videos or gradients before any CUDA call.
"""
import ctypes
import re

import pytest

from kccotgan_b200 import _lib
from test_footprint import _dump, _max_threads, _res_usage


@pytest.fixture(scope="module")
def lib():
    from kccotgan_b200 import build
    build.build()
    return _lib.load()


def _one(table, kernel):
    found = {n: v for n, v in table.items() if re.search(rf"\d{kernel}E", n)}
    assert len(found) == 1, f"{kernel}: {sorted(found)}"
    return next(iter(found.values()))


def test_bf16_gradient_kernel_fits_two_ctas_per_sm(lib):
    reg, stack, local = _one(_res_usage(), "grad_tc_bf16_kernel")
    threads = _one(_max_threads(), "grad_tc_bf16_kernel")
    assert reg * threads <= 32768, f"{reg} registers x {threads} threads"
    assert stack == 0 and local == 0, f"stack {stack}, local {local} bytes (spills)"


def test_bf16_distance_kernel_does_not_spill(lib):
    reg, stack, local = _one(_res_usage(), "sqdist_tc_bf16_kernel")
    assert stack == 0 and local == 0, f"stack {stack}, local {local} bytes (spills)"
    assert "sqdist_tc_bf16_kernel" in _dump("-symbols")


P = ctypes.c_void_p
GOOD = P(0x10000)                  # never dereferenced: every call below fails its argument check first


def _fwd(lib, real, fake, flags, B=8, K=128):
    return lib.kccot_mixed_loss_fwd_bf16(real, fake, 1, B, K, GOOD, GOOD, GOOD, GOOD, 2, 1, 1.0, 1.0, 1, GOOD, GOOD,
                                         None, GOOD, 1 << 20, flags, None, 0, 0)


def _bwd(lib, real, fake, g_real, g_fake, flags, B=8, K=128):
    return lib.kccot_mixed_loss_bwd_bf16(GOOD, real, fake, 1, B, K, GOOD, GOOD, GOOD, GOOD, 2, 1, 1.0, 1.0, 1, GOOD,
                                         g_real, g_fake, None, None, None, None, GOOD, 1 << 20, flags, None, 0, 0)


def test_accumulate_is_rejected(lib):
    assert _fwd(lib, GOOD, GOOD, _lib.FLAG_ACCUMULATE) == _lib.EINVAL
    assert "ACCUMULATE" in _lib.last_error()
    assert _bwd(lib, GOOD, GOOD, GOOD, GOOD, _lib.FLAG_ACCUMULATE) == _lib.EINVAL
    assert "ACCUMULATE" in _lib.last_error()


def test_misaligned_pointers_are_rejected(lib):
    bad = P(0x10002)
    assert _fwd(lib, bad, GOOD, 0) == _lib.EINVAL and "aligned" in _lib.last_error()
    assert _fwd(lib, GOOD, bad, 0) == _lib.EINVAL and "aligned" in _lib.last_error()
    for args in ((bad, GOOD, GOOD, GOOD), (GOOD, GOOD, bad, None), (GOOD, GOOD, None, bad)):
        assert _bwd(lib, *args, 0) == _lib.EINVAL and "aligned" in _lib.last_error()


def test_workspace_query(lib):
    # native shapes need no more than the fp32 call; widened shapes add the fp32 copies and gradient scratch
    for B, K in ((64, 122880), (32, 81920), (8, 128)):
        assert lib.kccot_mixed_loss_workspace_bytes_bf16(1, B, K, 100, 0) == lib.kccot_mixed_loss_workspace_bytes(1, B, K, 100)
    for B, K, flags in ((30, 1536, 0), (16, 300, 0), (32, 2048, _lib.PATH_SIMT), (128, 1024, 0)):
        extra = 4 * ((B * K * 4 + 255) // 256 * 256)
        assert lib.kccot_mixed_loss_workspace_bytes_bf16(1, B, K, 100, flags) == \
            lib.kccot_mixed_loss_workspace_bytes(1, B, K, 100) + extra
    assert lib.kccot_mixed_loss_workspace_bytes_bf16(0, 8, 128, 100, 0) == 0
