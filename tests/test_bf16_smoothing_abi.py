"""bf16 entry points of the Gaussian smoothing, host side and compiled footprint (no GPU needed).

Every argument error of kccot_smooth_fwd_bf16 / _bwd_bf16 (null pointers, the reference's '2d' mode, a radius above
6, an axis not longer than the radius, a misaligned tie mask, a short workspace) is reported before any CUDA call, with
the codes of the fp32 entries.  The tie mask holds one bit per element, rounded up to whole 32-bit words.  No bf16
smoothing kernel spills (read from the built library as in test_footprint.py).
"""
import ctypes
import re

import pytest

from kccotgan_b200 import _lib
from test_footprint import _res_usage

P = ctypes.c_void_p
GOOD = P(0x10000)                  # never dereferenced: every call below fails its argument check first
TAPS = (ctypes.c_float * 13)(*([1.0 / 13] * 13))


@pytest.fixture(scope="module")
def lib():
    from kccotgan_b200 import build
    build.build()
    return _lib.load()


def _fwd(lib, mode=1, x=GOOD, out=GOOD, maxval=GOOD, ties=GOOD, shape=(2, 8, 8, 8, 3), r=3, ws=GOOD, ws_bytes=1 << 30):
    return lib.kccot_smooth_fwd_bf16(mode, x, *shape, TAPS, r, TAPS, r, out, maxval, ties, ws, ws_bytes, None)


def _bwd(lib, mode=1, gout=GOOD, out=GOOD, maxval=GOOD, ties=GOOD, gx=GOOD, shape=(2, 8, 8, 8, 3), r=3, ws=GOOD,
         ws_bytes=1 << 30):
    return lib.kccot_smooth_bwd_bf16(mode, gout, out, maxval, ties, *shape, TAPS, r, TAPS, r, gx, ws, ws_bytes, None)


def test_ties_bytes(lib):
    for shape, words in (((1, 1, 1, 1, 1), 1), ((1, 1, 32, 1, 1), 1), ((1, 1, 33, 1, 1), 2), ((2, 9, 7, 10, 1), 40),
                         ((64, 64, 12, 64, 3), 64 * 64 * 12 * 64 * 3 // 32)):
        assert lib.kccot_smooth_ties_bytes(*shape) == 4 * words, shape
    assert lib.kccot_smooth_ties_bytes(0, 8, 8, 8, 1) == 0


def test_mode_errors(lib):
    assert _fwd(lib, mode=2) == _lib.EINVAL and "'2d'" in _lib.last_error()
    assert _bwd(lib, mode=2) == _lib.EINVAL and "mode" in _lib.last_error()


def test_null_pointers(lib):
    for kw in ({"x": None}, {"out": None}, {"maxval": None}, {"ties": None}):
        assert _fwd(lib, **kw) == _lib.EINVAL and "null" in _lib.last_error(), kw
    for kw in ({"gout": None}, {"out": None}, {"maxval": None}, {"ties": None}, {"gx": None}, {"ws": None}):
        assert _bwd(lib, **kw) == _lib.EINVAL and "null" in _lib.last_error(), kw
    with pytest.raises(ValueError, match="null"):
        _lib.call("kccot_smooth_fwd_bf16", 1, None, 2, 8, 8, 8, 3, TAPS, 3, TAPS, 3, None, None, None, None, 0, None)


def test_misaligned_tie_mask(lib):
    for call in (_fwd, _bwd):
        assert call(lib, ties=P(0x10002)) == _lib.EINVAL and "aligned" in _lib.last_error()


def test_radius_and_axis_limits(lib):
    for call in (_fwd, _bwd):
        for mode in (1, 3):
            assert call(lib, mode=mode, r=7) == _lib.EUNSUPPORTED and "radius 7" in _lib.last_error()
            assert call(lib, mode=mode, r=0) == _lib.EUNSUPPORTED
        assert call(lib, mode=1, shape=(2, 8, 3, 8, 3)) == _lib.EINVAL and "T > 3" in _lib.last_error()
        assert call(lib, mode=1, shape=(2, 8, 1025, 8, 3)) == _lib.EINVAL and "1024" in _lib.last_error()
        assert call(lib, mode=3, shape=(2, 3, 8, 8, 3)) == _lib.EINVAL and "H, W > 3" in _lib.last_error()
        assert call(lib, mode=3, shape=(2, 8, 8, 2, 3), r=2) == _lib.EINVAL and "H, W > 2" in _lib.last_error()
        assert call(lib, mode=1, shape=(0, 8, 8, 8, 3)) == _lib.EINVAL and "sizes" in _lib.last_error()


def test_workspace(lib):
    need = lib.kccot_smooth_workspace_bytes(3, 2, 8, 8, 8, 3)
    for call in (_fwd, _bwd):
        assert call(lib, mode=3, ws_bytes=need - 256) == _lib.EINVAL and "workspace" in _lib.last_error()
    assert _fwd(lib, mode=3, ws=None) == _lib.EINVAL


def test_bf16_smoothing_kernels_do_not_spill(lib):
    usage = _res_usage()
    found = {n: v for n, v in usage.items()
             if re.search(r"\d(axis_col_bf16_kernel|axis_tile_bf16_kernel|tie_sums_bf16_kernel)", n)}
    # 7 passes (forward: 2 in mode 1, 2 in mode 3; backward: 1 and 2) x 6 radii x (tile kernel, column kernels of 8,
    # 4 and 1 elements per thread), and the tie sums
    assert len(found) == 7 * 6 * 4 + 1, len(found)
    spills = {n: v for n, v in found.items() if v[1] or v[2]}
    assert not spills, spills
