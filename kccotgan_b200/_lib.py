"""ctypes binding of libkccot.so (the C ABI in include/kccot.h).

There is NO fallback: if the shared library is missing or the device is not a B200 the import /
first call raises.  Build with `python -m kccotgan_b200.build`.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkccot.so")

PATH_AUTO, PATH_SIMT, PATH_TCGEN05, FLAG_ACCUMULATE = 0, 1, 2, 16
SHARD_FLAGS_PER_RANK = 256          # KCCOT_SHARD_FLAGS_PER_RANK of include/kccot.h
EINVAL, ECUDA, EWORKSPACE, EUNSUPPORTED = -1, -2, -3, -4

_c = ctypes
_P, _I, _LL, _F, _SZ = _c.c_void_p, _c.c_int, _c.c_longlong, _c.c_float, _c.c_size_t

# name -> (restype, argtypes); mirrors include/kccot.h one to one
SIGNATURES = {
    "kccot_version": (_I, []),
    "kccot_last_error": (_c.c_char_p, []),
    "kccot_device_check": (_I, []),
    "kccot_launch_count": (_c.c_ulonglong, []),
    "kccot_cost_workspace_bytes": (_SZ, [_I, _I, _I, _LL]),
    "kccot_cost_fwd": (_I, [_P, _P, _I, _I, _I, _LL, _P, _P, _P, _P, _I, _I, _F, _P, _P, _SZ, _I, _P]),
    "kccot_mixed_cost_workspace_bytes": (_SZ, [_I, _I, _LL]),
    "kccot_mixed_cost_fwd": (_I, [_P, _P, _I, _I, _LL, _P, _P, _P, _P, _I, _I, _F, _P, _P, _SZ, _I, _P]),
    "kccot_mixed_sqdist_partials": (_I, [_P, _P, _I, _I, _LL, _P, _SZ, _I, _P]),
    "kccot_cost_bwd_workspace_bytes": (_SZ, [_I, _I, _I, _LL]),
    "kccot_cost_bwd": (_I, [_P, _P, _P, _I, _I, _I, _LL, _F, _P, _P, _P, _SZ, _I, _P]),
    "kccot_martingale_bwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _F, _P, _P, _I, _P]),
    "kccot_mixed_cost_bwd_workspace_bytes": (_SZ, [_I, _I, _LL]),
    "kccot_mixed_cost_bwd": (_I, [_P, _P, _P, _I, _I, _LL, _P, _P, _P, _P, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P,
                                  _SZ, _I, _P]),
    "kccot_sinkhorn_workspace_bytes": (_SZ, [_I, _I, _I]),
    "kccot_sinkhorn_fwd": (_I, [_P, _I, _I, _F, _I, _I, _F, _I, _P, _P, _P, _P, _P, _SZ, _P]),
    "kccot_sinkhorn_bwd": (_I, [_P, _I, _I, _F, _I, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "kccot_shard_cost_workspace_bytes": (_SZ, [_I, _LL, _I]),
    "kccot_shard_cost_fwd": (_I, [_P, _P, _I, _LL, _I, _I, _P, _P, _P, _P, _I, _I, _F, _P, _P, _SZ, _P]),
    "kccot_shard_cost_bwd": (_I, [_P, _P, _P, _I, _LL, _I, _I, _P, _P, _P, _P, _I, _I, _F, _P, _P, _P, _P, _P, _P, _SZ,
                                  _P]),
    "kccot_shard_cost_fwd_bf16": (_I, [_P, _P, _I, _LL, _I, _I, _P, _P, _P, _P, _I, _I, _F, _P, _P, _SZ, _P]),
    "kccot_shard_cost_bwd_bf16": (_I, [_P, _P, _P, _I, _LL, _I, _I, _P, _P, _P, _P, _I, _I, _F, _P, _P, _P, _P, _P, _P,
                                       _SZ, _P]),
    "kccot_shard_cost_workspace_bytes_ctx": (_SZ, [_I, _LL, _I, _LL, _LL]),
    "kccot_shard_cost_fwd_ctx": (_I, [_P, _P, _I, _LL, _I, _I, _P, _P, _P, _P, _I, _I, _F, _P, _P, _SZ, _P, _LL, _LL]),
    "kccot_shard_cost_bwd_ctx": (_I, [_P, _P, _P, _I, _LL, _I, _I, _P, _P, _P, _P, _I, _I, _F, _P, _P, _P, _P, _P, _P,
                                      _SZ, _P, _LL, _LL]),
    "kccot_shard_cost_fwd_bf16_ctx": (_I, [_P, _P, _I, _LL, _I, _I, _P, _P, _P, _P, _I, _I, _F, _P, _P, _SZ, _P, _LL,
                                           _LL]),
    "kccot_shard_cost_bwd_bf16_ctx": (_I, [_P, _P, _P, _I, _LL, _I, _I, _P, _P, _P, _P, _I, _I, _F, _P, _P, _P, _P, _P,
                                           _P, _SZ, _P, _LL, _LL]),
    "kccot_shard_sinkhorn_workspace_bytes": (_SZ, [_I, _I, _I, _I]),
    "kccot_shard_mailbox_bytes": (_SZ, [_I, _I, _I]),
    "kccot_shard_local_min": (_I, [_P, _I, _I, _I, _P, _P]),
    "kccot_shard_sinkhorn_fwd": (_I, [_P, _I, _I, _I, _I, _F, _I, _I, _F, _I, _P, _P, _P, _P, _P, _I, _I, _P, _P,
                                      _c.c_ulonglong, _P, _SZ, _P]),
    "kccot_shard_sinkhorn_bwd": (_I, [_P, _I, _I, _I, _I, _F, _I, _P, _P, _P, _P, _P, _P, _I, _I, _P, _P,
                                      _c.c_ulonglong, _P, _SZ, _P]),
    "kccot_mixed_loss_saved_bytes": (_SZ, [_I, _I, _I]),
    "kccot_mixed_loss_workspace_bytes": (_SZ, [_I, _I, _LL, _I]),
    "kccot_mixed_loss_fwd": (_I, [_P, _P, _I, _I, _LL, _P, _P, _P, _P, _I, _I, _F, _F, _I, _P, _P, _P, _P, _SZ, _I, _P]),
    "kccot_mixed_loss_bwd": (_I, [_P, _P, _P, _I, _I, _LL, _P, _P, _P, _P, _I, _I, _F, _F, _I, _P, _P, _P, _P, _P, _P,
                                  _P, _P, _SZ, _I, _P]),
    "kccot_mixed_loss_fwd_ctx": (_I, [_P, _P, _I, _I, _LL, _P, _P, _P, _P, _I, _I, _F, _F, _I, _P, _P, _P, _P, _SZ, _I, _P,
                                      _LL, _LL]),
    "kccot_mixed_loss_bwd_ctx": (_I, [_P, _P, _P, _I, _I, _LL, _P, _P, _P, _P, _I, _I, _F, _F, _I, _P, _P, _P, _P, _P, _P,
                                      _P, _P, _SZ, _I, _P, _LL, _LL]),
    "kccot_mixed_loss_workspace_bytes_bf16": (_SZ, [_I, _I, _LL, _I, _I]),
    "kccot_mixed_loss_fwd_bf16": (_I, [_P, _P, _I, _I, _LL, _P, _P, _P, _P, _I, _I, _F, _F, _I, _P, _P, _P, _P, _SZ, _I,
                                       _P, _LL, _LL]),
    "kccot_mixed_loss_bwd_bf16": (_I, [_P, _P, _P, _I, _I, _LL, _P, _P, _P, _P, _I, _I, _F, _F, _I, _P, _P, _P, _P, _P,
                                       _P, _P, _P, _SZ, _I, _P, _LL, _LL]),
    "kccot_pm_fwd": (_I, [_P, _I, _I, _I, _F, _F, _P, _P, _P]),
    "kccot_pm_bwd": (_I, [_P, _I, _I, _I, _F, _F, _P, _P, _P, _P]),
    "kccot_pm_batched_fwd": (_I, [_P, _I, _I, _I, _I, _F, _F, _P, _P, _P]),
    "kccot_pm_batched_bwd": (_I, [_P, _I, _I, _I, _I, _F, _F, _P, _P, _P, _P]),
    "kccot_smooth_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I, _I]),
    "kccot_smooth_fwd": (_I, [_I, _P, _I, _I, _I, _I, _I, _P, _I, _P, _I, _P, _P, _P, _SZ, _P]),
    "kccot_smooth_bwd": (_I, [_I, _P, _P, _P, _I, _I, _I, _I, _I, _P, _I, _P, _I, _P, _P, _SZ, _P]),
    "kccot_smooth_ties_bytes": (_SZ, [_I, _I, _I, _I, _I]),
    "kccot_smooth_fwd_bf16": (_I, [_I, _P, _I, _I, _I, _I, _I, _P, _I, _P, _I, _P, _P, _P, _P, _SZ, _P]),
    "kccot_smooth_bwd_bf16": (_I, [_I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _I, _P, _I, _P, _P, _SZ, _P]),
    "kccot_smooth_fwd_dev": (_I, [_I, _P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _P, _SZ, _P]),
    "kccot_smooth_bwd_dev": (_I, [_I, _P, _P, _P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _SZ, _P]),
    "kccot_smooth_fwd_bf16_dev": (_I, [_I, _P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _P, _P, _SZ, _P]),
    "kccot_smooth_bwd_bf16_dev": (_I, [_I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _SZ, _P]),
    "kccot_smooth_batched_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I, _I, _I]),
    "kccot_smooth_batched_fwd": (_I, [_I, _P, _I, _I, _I, _I, _I, _I, _P, _I, _P, _P, _P, _SZ, _P]),
    "kccot_smooth_batched_bwd": (_I, [_I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _I, _P, _P, _SZ, _P]),
    "kccot_smooth_batched_fwd_bf16": (_I, [_I, _P, _I, _I, _I, _I, _I, _I, _P, _I, _P, _P, _P, _P, _SZ, _P]),
    "kccot_smooth_batched_bwd_bf16": (_I, [_I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _I, _P, _P, _SZ, _P]),
}

_lib = None


def load():
    """Load libkccot.so (once).  Raises OSError with build instructions if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise OSError(f"{LIB_PATH} not found: build the CUDA library with `python -m kccotgan_b200.build` "
                          "(kccotgan_b200 has no CPU or PyTorch fallback)")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if lib.kccot_version() != 203:
            raise OSError(f"{LIB_PATH}: ABI version {lib.kccot_version()} != 203; rebuild")
        _lib = lib
    return _lib


def last_error():
    return load().kccot_last_error().decode("utf-8", "replace")


def check(rc):
    """Map an ABI return code onto the exception type the reference's callers would see."""
    if rc == 0:
        return
    msg = last_error()
    if rc == EINVAL:
        raise ValueError(f"kccot: {msg}")
    raise RuntimeError(f"kccot (code {rc}): {msg}")


def call(name, *args):
    check(getattr(load(), name)(*args))
