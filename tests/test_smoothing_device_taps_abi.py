"""Device-weight entry points of the Gaussian smoothing, host side (no GPU needed).

kccot_smooth_fwd_dev / _bwd_dev / _fwd_bf16_dev / _bwd_bf16_dev take the 2r+1 weights as a device array instead of
host arrays.  Every argument error (a null or misaligned weight array, a radius outside 1..6, the reference's '2d'
mode, an axis not longer than the radius) is reported before any CUDA call, with the codes of the host-weight entries.
A data_utils.SmoothingTaps of the wrong radius, or a CPU video, raises ValueError before anything reaches the device.
"""
import ctypes

import pytest
import torch

from kccotgan_b200 import _lib

P = ctypes.c_void_p
GOOD = P(0x10000)                  # never dereferenced: every call below fails its argument check first
SHAPE = (2, 8, 8, 8, 3)


@pytest.fixture(scope="module")
def lib():
    from kccotgan_b200 import build
    build.build()
    return _lib.load()


def _fwd(lib, mode=1, taps=GOOD, r=3, shape=SHAPE):
    return lib.kccot_smooth_fwd_dev(mode, GOOD, *shape, taps, r, GOOD, GOOD, GOOD, 1 << 30, None)


def _bwd(lib, mode=1, taps=GOOD, r=3, shape=SHAPE):
    return lib.kccot_smooth_bwd_dev(mode, GOOD, GOOD, GOOD, *shape, taps, r, GOOD, GOOD, 1 << 30, None)


def _fwd_bf16(lib, mode=1, taps=GOOD, r=3, shape=SHAPE):
    return lib.kccot_smooth_fwd_bf16_dev(mode, GOOD, *shape, taps, r, GOOD, GOOD, GOOD, GOOD, 1 << 30, None)


def _bwd_bf16(lib, mode=1, taps=GOOD, r=3, shape=SHAPE):
    return lib.kccot_smooth_bwd_bf16_dev(mode, GOOD, GOOD, GOOD, GOOD, *shape, taps, r, GOOD, GOOD, 1 << 30, None)


ENTRIES = [_fwd, _bwd, _fwd_bf16, _bwd_bf16]


@pytest.mark.parametrize("call", ENTRIES)
def test_weight_array_errors(lib, call):
    for mode in (1, 3):
        assert call(lib, mode=mode, taps=None) == _lib.EINVAL and "null weights" in _lib.last_error()
        for addr in (0x10001, 0x10002, 0x10003):
            assert call(lib, mode=mode, taps=P(addr)) == _lib.EINVAL and "aligned" in _lib.last_error(), addr


@pytest.mark.parametrize("call", ENTRIES)
def test_radius_mode_and_axis_errors(lib, call):
    for mode in (1, 3):
        assert call(lib, mode=mode, r=7) == _lib.EUNSUPPORTED and "radius 7" in _lib.last_error()
        assert call(lib, mode=mode, r=0) == _lib.EUNSUPPORTED and "radius 0" in _lib.last_error()
    assert call(lib, mode=2) == _lib.EINVAL and "mode" in _lib.last_error()
    assert call(lib, mode=1, shape=(2, 8, 3, 8, 3)) == _lib.EINVAL and "T > 3" in _lib.last_error()
    assert call(lib, mode=3, shape=(2, 8, 3, 8, 3)) == _lib.EINVAL and "T > 3" in _lib.last_error()
    assert call(lib, mode=3, shape=(2, 3, 8, 8, 3)) == _lib.EINVAL and "H, W > 3" in _lib.last_error()
    assert call(lib, mode=3, shape=(2, 8, 8, 2, 3), r=2) == _lib.EINVAL and "H, W > 2" in _lib.last_error()


def test_smoothing_taps_radius_must_match():
    from kccotgan_b200.data_utils import KernelSmoothing, SmoothingTaps
    ks = KernelSmoothing(temporal_kernel_size=6, spatial_kernel_size=8)        # radii 3 and 4
    x = torch.rand(2, 8, 6, 8, 1)
    with pytest.raises(ValueError, match="radius 4 for a filter of radius 3"):
        ks.temporal_convolution(x, SmoothingTaps(4, device="cpu"))
    with pytest.raises(ValueError, match="radius 3 for a filter of radius 4"):
        ks.gaussian_convolution3D(x, SmoothingTaps(3, device="cpu"))


def test_smoothing_taps_cpu_video_raises():
    from kccotgan_b200.data_utils import KernelSmoothing, SmoothingTaps
    ks = KernelSmoothing(temporal_kernel_size=6, spatial_kernel_size=6)
    taps = SmoothingTaps(3, device="cpu").set(2.0)
    for dtype in (torch.float32, torch.bfloat16):
        x = torch.rand(2, 8, 6, 8, 1).to(dtype)
        for fn in (ks.temporal_convolution, ks.gaussian_convolution3D):
            with pytest.raises(ValueError, match="CUDA"):
                fn(x, taps)


def test_smoothing_taps_set_writes_the_host_weights():
    from kccotgan_b200.data_utils import KernelSmoothing, SmoothingTaps
    taps = SmoothingTaps(3, device="cpu")
    for sigma in (5.0, 0.7, KernelSmoothing().annealing_sigma(5.0, 12345)):
        assert taps.set(sigma) is taps
        assert torch.equal(taps.weights, torch.from_numpy(KernelSmoothing._weights(3, sigma)))
