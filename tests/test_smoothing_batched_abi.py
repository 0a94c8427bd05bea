"""Batched entry points of the Gaussian smoothing, host side and compiled footprint (no GPU needed).

kccot_smooth_batched_fwd / _bwd / _fwd_bf16 / _bwd_bf16 smooth nprob independent videos in one call.  Every argument
error (those of the *_dev entries, plus a problem count outside 1..65535, a short or misaligned workspace) is reported
before any CUDA call, with the codes of the single-problem entries.  The workspace holds 2 * nprob tie sums and, in
mode 3, two fp32 intermediates of the whole batch.  No batched smoothing kernel spills.  SmoothingTaps(r, nprob=...)
writes one row of weights per problem, and the batched Python methods reject bad inputs before anything reaches the
device.
"""
import ctypes
import re

import pytest
import torch

from kccotgan_b200 import _lib
from test_footprint import _res_usage

P = ctypes.c_void_p
GOOD = P(0x10000)                  # never dereferenced: every call below fails its argument check first
SHAPE = (2, 8, 8, 8, 3)


@pytest.fixture(scope="module")
def lib():
    from kccotgan_b200 import build
    build.build()
    return _lib.load()


def _fwd(lib, mode=1, nprob=3, x=GOOD, out=GOOD, maxval=GOOD, taps=GOOD, r=3, shape=SHAPE, ws=GOOD, ws_bytes=1 << 30):
    return lib.kccot_smooth_batched_fwd(mode, x, nprob, *shape, taps, r, out, maxval, ws, ws_bytes, None)


def _bwd(lib, mode=1, nprob=3, gout=GOOD, out=GOOD, maxval=GOOD, gx=GOOD, taps=GOOD, r=3, shape=SHAPE, ws=GOOD,
         ws_bytes=1 << 30):
    return lib.kccot_smooth_batched_bwd(mode, gout, out, maxval, nprob, *shape, taps, r, gx, ws, ws_bytes, None)


def _fwd_bf16(lib, mode=1, nprob=3, x=GOOD, out=GOOD, maxval=GOOD, ties=GOOD, taps=GOOD, r=3, shape=SHAPE, ws=GOOD,
              ws_bytes=1 << 30):
    return lib.kccot_smooth_batched_fwd_bf16(mode, x, nprob, *shape, taps, r, out, maxval, ties, ws, ws_bytes, None)


def _bwd_bf16(lib, mode=1, nprob=3, gout=GOOD, out=GOOD, maxval=GOOD, ties=GOOD, gx=GOOD, taps=GOOD, r=3,
              shape=SHAPE, ws=GOOD, ws_bytes=1 << 30):
    return lib.kccot_smooth_batched_bwd_bf16(mode, gout, out, maxval, ties, nprob, *shape, taps, r, gx, ws, ws_bytes,
                                             None)


ENTRIES = [_fwd, _bwd, _fwd_bf16, _bwd_bf16]
POINTERS = {_fwd: ("x", "out", "maxval"), _bwd: ("gout", "out", "maxval", "gx", "ws"),
            _fwd_bf16: ("x", "out", "maxval", "ties"), _bwd_bf16: ("gout", "out", "maxval", "ties", "gx", "ws")}


@pytest.fixture(autouse=True)
def _no_launch(request):
    """every test here fails before any CUDA call: the library's launch counter does not move"""
    if "lib" not in request.fixturenames:
        yield
        return
    lib = request.getfixturevalue("lib")
    before = lib.kccot_launch_count()
    yield
    assert lib.kccot_launch_count() == before


@pytest.mark.parametrize("call", ENTRIES)
def test_mode_and_null_pointers(lib, call):
    assert call(lib, mode=2) == _lib.EINVAL and "mode" in _lib.last_error()
    for name in POINTERS[call]:
        assert call(lib, **{name: None}) == _lib.EINVAL and "null" in _lib.last_error(), name


@pytest.mark.parametrize("call", ENTRIES)
def test_problem_count(lib, call):
    for nprob in (0, -1, 65536):
        assert call(lib, nprob=nprob) == _lib.EINVAL and "nprob" in _lib.last_error(), nprob


@pytest.mark.parametrize("call", ENTRIES)
def test_weight_array_errors(lib, call):
    for mode in (1, 3):
        assert call(lib, mode=mode, taps=None) == _lib.EINVAL and "null weights" in _lib.last_error()
        for addr in (0x10001, 0x10002, 0x10003):
            assert call(lib, mode=mode, taps=P(addr)) == _lib.EINVAL and "aligned" in _lib.last_error(), addr


@pytest.mark.parametrize("call", ENTRIES)
def test_radius_and_axis_errors(lib, call):
    for mode in (1, 3):
        assert call(lib, mode=mode, r=7) == _lib.EUNSUPPORTED and "radius 7" in _lib.last_error()
        assert call(lib, mode=mode, r=0) == _lib.EUNSUPPORTED and "radius 0" in _lib.last_error()
    assert call(lib, mode=1, shape=(2, 8, 3, 8, 3)) == _lib.EINVAL and "T > 3" in _lib.last_error()
    assert call(lib, mode=3, shape=(2, 8, 3, 8, 3)) == _lib.EINVAL and "T > 3" in _lib.last_error()
    assert call(lib, mode=3, shape=(2, 3, 8, 8, 3)) == _lib.EINVAL and "H, W > 3" in _lib.last_error()
    assert call(lib, mode=3, shape=(2, 8, 8, 2, 3), r=2) == _lib.EINVAL and "H, W > 2" in _lib.last_error()
    assert call(lib, mode=1, shape=(2, 8, 1025, 8, 3)) == _lib.EINVAL and "1024" in _lib.last_error()
    assert call(lib, mode=1, shape=(0, 8, 8, 8, 3)) == _lib.EINVAL and "sizes" in _lib.last_error()


@pytest.mark.parametrize("call", [_fwd_bf16, _bwd_bf16])
def test_misaligned_tie_mask(lib, call):
    assert call(lib, ties=P(0x10002)) == _lib.EINVAL and "aligned" in _lib.last_error()


@pytest.mark.parametrize("call", ENTRIES)
def test_workspace_errors(lib, call):
    nprob = 40                                   # more sums than the 256-byte head of the single-problem call holds
    for mode in (1, 3) if call in (_bwd, _bwd_bf16) else (3,):          # the mode-1 forward uses no workspace
        need = lib.kccot_smooth_batched_workspace_bytes(mode, nprob, *SHAPE)
        assert call(lib, mode=mode, nprob=nprob, ws_bytes=need - 1) == _lib.EINVAL and "workspace" in _lib.last_error()
        assert call(lib, mode=mode, nprob=nprob, ws=None) == _lib.EINVAL
        assert call(lib, mode=mode, nprob=nprob, ws=P(0x10004)) == _lib.EINVAL and "aligned" in _lib.last_error()


def test_workspace_bytes(lib):
    for mode in (1, 3):
        for shape in (SHAPE, (64, 32, 10, 32, 1), (2, 14, 9, 65, 1)):
            single = lib.kccot_smooth_workspace_bytes(mode, *shape)
            sizes = [lib.kccot_smooth_batched_workspace_bytes(mode, nprob, *shape) for nprob in (1, 2, 32, 33, 256)]
            assert sizes[0] >= single, (mode, shape)
            assert all(b > a for a, b in zip(sizes, sizes[1:])) or mode == 1, (mode, shape, sizes)
            assert all(b >= a for a, b in zip(sizes, sizes[1:])), (mode, shape, sizes)
            n = 1
            for v in shape:
                n *= v
            for nprob, size in zip((1, 2, 32, 33, 256), sizes):
                assert size >= 2 * nprob * 4 + (2 * nprob * n * 4 if mode == 3 else 0), (mode, nprob, size)
    # room for the sums: one 256-byte head holds 32 problems, 33 need a second
    assert lib.kccot_smooth_batched_workspace_bytes(1, 33, *SHAPE) > lib.kccot_smooth_batched_workspace_bytes(1, 32,
                                                                                                             *SHAPE)
    assert lib.kccot_smooth_batched_workspace_bytes(1, 0, *SHAPE) == 0


def test_batched_smoothing_kernels_do_not_spill(lib):
    found = {n: v for n, v in _res_usage().items()
             if re.search(r"\d(axis_col_batched_kernel|axis_tile_batched_kernel|tie_sums_batched_kernel)", n)}
    # tile and column kernels of every pass of both dtypes and radii 1..6, and the fp32 and bf16 tie sums
    assert len(found) > 2 * 6 * 2, len(found)
    spills = {n: v for n, v in found.items() if v[1] or v[2]}
    assert not spills, spills


def test_smoothing_taps_rows():
    from kccotgan_b200.data_utils import KernelSmoothing, SmoothingTaps
    taps = SmoothingTaps(3, device="cpu", nprob=3)
    assert tuple(taps.weights.shape) == (3, 7)
    sig = [5.0, 0.7, KernelSmoothing().annealing_sigma(5.0, 12345)]
    assert taps.set(sig) is taps
    for p, s in enumerate(sig):
        assert torch.equal(taps.weights[p], torch.from_numpy(KernelSmoothing._weights(3, s))), p
    taps.set(2.0)
    for p in range(3):
        assert torch.equal(taps.weights[p], torch.from_numpy(KernelSmoothing._weights(3, 2.0))), p
    with pytest.raises(ValueError, match="2 sigmas for 3 problems"):
        taps.set([1.0, 2.0])
    with pytest.raises(ValueError, match="nprob"):
        SmoothingTaps(3, device="cpu", nprob=0)
    assert tuple(SmoothingTaps(3, device="cpu").weights.shape) == (7,)       # without nprob: as before


def test_batched_methods_reject_bad_inputs():
    from kccotgan_b200.data_utils import KernelSmoothing, SmoothingTaps
    ks = KernelSmoothing(temporal_kernel_size=6, spatial_kernel_size=6)
    x = torch.rand(3, 2, 8, 6, 8, 1)
    for fn in (ks.temporal_convolution_batched, ks.gaussian_convolution3D_batched):
        with pytest.raises(ValueError, match="CUDA"):
            fn(x, 2.0)
        with pytest.raises(ValueError, match="CUDA"):
            fn(x, SmoothingTaps(3, device="cpu", nprob=3).set(2.0))
        with pytest.raises(ValueError, match="radius 4 for a filter of radius 3"):
            fn(x, SmoothingTaps(4, device="cpu", nprob=3))
        with pytest.raises(ValueError, match="2 problems for a batch of 3"):
            fn(x, SmoothingTaps(3, device="cpu", nprob=2))
