"""Shared-context entry points of the row-sharded cost, host side (no GPU needed).

Every bad hint, null pointer, bad row range and misaligned bf16 pointer is rejected with KCCOT_EINVAL before any CUDA
call (on a box without a device any CUDA call would fail with KCCOT_ECUDA instead).  The workspace query without a hint
is the plain one.  The hinted pre-pass kernels do not spill.  ShardedMixedLoss checks `ctx_frames` before it touches a
device.
"""
import ctypes

import pytest

from kccotgan_b200 import _lib
from test_footprint import _res_usage


@pytest.fixture(scope="module")
def lib():
    from kccotgan_b200 import build
    build.build()
    return _lib.load()


P = ctypes.c_void_p
GOOD = P(0x10000)                  # never dereferenced: every call below fails its argument check first
BAD = P(0x10002)
B, K = 8, 4 * 16 * 16              # [B, H=4, T=16, W=16, C=1]: period 256
BAD_HINTS = [(256, -1), (-256, 16), (256, 256), (256, 300), (0, 16), (200, 16), (3 * K, 16)]


def _fwd(lib, name="kccot_shard_cost_fwd_ctx", real=GOOD, fake=GOOD, h=GOOD, row0=0, Brows=8, ws=GOOD, hint=(256, 16)):
    return getattr(lib, name)(real, fake, B, K, row0, Brows, h, GOOD, GOOD, GOOD, 2, 1, 1.0, GOOD, ws, 1 << 20, None,
                              *hint)


def _bwd(lib, name="kccot_shard_cost_bwd_ctx", g=GOOD, cbar=GOOD, row0=0, Brows=8, hint=(256, 16)):
    return getattr(lib, name)(cbar, GOOD, GOOD, B, K, row0, Brows, GOOD, GOOD, GOOD, GOOD, 2, 1, 1.0, g, GOOD, GOOD,
                              GOOD, GOOD, GOOD, 1 << 20, None, *hint)


FWD = ["kccot_shard_cost_fwd_ctx", "kccot_shard_cost_fwd_bf16_ctx"]
BWD = ["kccot_shard_cost_bwd_ctx", "kccot_shard_cost_bwd_bf16_ctx"]


@pytest.mark.parametrize("hint", BAD_HINTS, ids=str)
def test_bad_hints_are_rejected(lib, hint):
    for f in FWD:
        assert _fwd(lib, f, hint=hint) == _lib.EINVAL and "shared-context" in _lib.last_error(), (f, hint)
    for f in BWD:
        assert _bwd(lib, f, hint=hint) == _lib.EINVAL and "shared-context" in _lib.last_error(), (f, hint)
    assert lib.kccot_shard_cost_workspace_bytes_ctx(B, K, 8, *hint) == 0


def test_null_pointers_are_rejected(lib):
    for f in FWD:
        for kw in ({"real": None}, {"fake": None}, {"h": None}, {"ws": None}):
            assert _fwd(lib, f, **kw) == _lib.EINVAL and "null" in _lib.last_error(), (f, kw)
    for f in BWD:
        assert _bwd(lib, f, cbar=None) == _lib.EINVAL and "null" in _lib.last_error(), f


def test_misaligned_bf16_pointers_are_rejected(lib):
    assert _fwd(lib, FWD[1], real=BAD) == _lib.EINVAL and "aligned" in _lib.last_error()
    assert _fwd(lib, FWD[1], fake=BAD) == _lib.EINVAL and "aligned" in _lib.last_error()
    assert _bwd(lib, BWD[1], g=BAD) == _lib.EINVAL and "aligned" in _lib.last_error()


@pytest.mark.parametrize("row0, Brows", [(-1, 4), (0, 0), (6, 4), (8, 1)])
def test_bad_row_range_is_rejected(lib, row0, Brows):
    for f in FWD:
        assert _fwd(lib, f, row0=row0, Brows=Brows) == _lib.EINVAL and "row range" in _lib.last_error(), f
    for f in BWD:
        assert _bwd(lib, f, row0=row0, Brows=Brows) == _lib.EINVAL and "row range" in _lib.last_error(), f


@pytest.mark.parametrize("Bq, Kq, Brows, period", [(256, 1024, 256, 256), (128, 300, 64, 60), (96, 105, 96, 35),
                                                   (8192, 81920, 8192, 4096)])
def test_workspace_query(lib, Bq, Kq, Brows, period):
    plain = lib.kccot_shard_cost_workspace_bytes(Bq, Kq, Brows)
    assert plain > 0
    assert lib.kccot_shard_cost_workspace_bytes_ctx(Bq, Kq, Brows, 0, 0) == plain
    assert lib.kccot_shard_cost_workspace_bytes_ctx(Bq, Kq, Brows, period, 0) == plain
    hinted = lib.kccot_shard_cost_workspace_bytes_ctx(Bq, Kq, Brows, period, period // 2)
    # the permuted split is at most one 64-column tile wider; the predicted-column gradient rows come on top
    assert hinted >= plain + Brows * (Kq - Kq // period * (period // 2)) * 4
    assert hinted <= plain + Brows * Kq * 4 + 4 * (2 * Bq + 64) * 64 * 2 + 4096


@pytest.mark.parametrize("kernel", ["colsum_part_ctx_kernel", "split_ctx_kernel", "ctx_scatter_kernel"])
def test_ctx_kernels_do_not_spill(lib, kernel):
    usage = _res_usage()
    found = [(n, v) for n, v in usage.items() if kernel in n]
    assert len(found) == 2, sorted(usage)                  # fp32 and bf16 instantiations
    for n, (reg, stack, local) in found:
        assert stack == 0 and local == 0, f"{n}: stack {stack}, local {local} bytes (spills)"


def test_sharded_loss_checks_ctx_frames_first():
    from kccotgan_b200.sharded import ShardedMixedLoss
    for bad in (-1, 4, 5):
        with pytest.raises(ValueError, match="ctx_frames"):
            ShardedMixedLoss(256, 1024, 4, 8, 1.0, ctx_frames=bad)
    with pytest.raises(ValueError, match="backend"):
        ShardedMixedLoss(256, 1024, 4, 8, 1.0, ctx_frames=1, backend=object())
