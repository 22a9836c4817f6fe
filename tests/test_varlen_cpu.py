"""CPU tests of the packed variable-length attention symbols: NULL handles and num_seqs == 0 are argument errors, and
without a device the calls report MFA_ERROR_DEVICE_NOT_SUPPORTED -- never a crash, never a CPU fallback."""
import ctypes

import numpy as np
import pytest

INVALID_ARGS, DEVICE_NOT_SUPPORTED = 1, 3


def _fwd(lib, ctx, bufs, cu, num_seqs):
    return lib.mfa_attention_forward_varlen(ctx, *bufs, cu, cu, num_seqs, 8, 8, 2, 1, 64, 0.125, True, -1, 1, 2, None)


def _bwd(lib, ctx, bufs, cu, num_seqs):
    return lib.mfa_attention_backward_varlen(ctx, *bufs, cu, cu, num_seqs, 8, 8, 2, 1, 64, 0.125, True, -1, 1, None)


def test_varlen_null_handles_and_empty_batches_are_invalid_args():
    from umfa import _ffi
    lib = _ffi._lib
    assert _fwd(lib, None, [None] * 5, None, 1) == INVALID_ARGS
    assert _bwd(lib, None, [None] * 10, None, 1) == INVALID_ARGS
    # handles the library must not dereference before these checks: placeholders over zeroed memory
    keep = np.zeros(4096, np.uint8)
    h = ctypes.c_void_p(keep.ctypes.data)
    assert _fwd(lib, h, [h] * 5, None, 2) == INVALID_ARGS           # NULL cu_seqlens
    assert _fwd(lib, h, [h] * 5, h, 0) == INVALID_ARGS              # num_seqs == 0
    assert _bwd(lib, h, [h] * 10, h, 0) == INVALID_ARGS
    assert _bwd(lib, h, [None] + [h] * 9, h, 2) == INVALID_ARGS     # NULL dout


def test_varlen_without_device_reports_it():
    import umfa
    from umfa import _ffi
    if umfa.is_metal_available():
        pytest.skip("a GPU is present")
    lib = _ffi._lib
    keep = np.zeros(4096, np.uint8)
    h = ctypes.c_void_p(keep.ctypes.data)
    assert _fwd(lib, h, [h] * 5, h, 2) == DEVICE_NOT_SUPPORTED
    assert _bwd(lib, h, [h] * 10, h, 2) == DEVICE_NOT_SUPPORTED
    assert _fwd(lib, h, [h, h, h, h, None], h, 2) == DEVICE_NOT_SUPPORTED      # lse is optional in the forward


def test_umfa_varlen_argument_validation():
    from umfa import core
    q = np.zeros((10, 4, 8), np.float32)
    k = np.zeros((12, 2, 8), np.float32)
    cu_q, cu_k = np.array([0, 4, 10]), np.array([0, 5, 12])
    assert core._varlen_dims(q, k, k, cu_q, cu_k, "thd")[:5] == (4, 2, 10, 12, 8)
    with pytest.raises(ValueError):
        core._varlen_dims(q, np.zeros((12, 3, 8), np.float32), np.zeros((12, 3, 8), np.float32), cu_q, cu_k, "thd")
    with pytest.raises(ValueError):
        core._varlen_dims(q, k, k, cu_q, cu_k[:2], "thd")
    with pytest.raises(ValueError):
        core._varlen_dims(q, k, k, cu_q, cu_k, "bshd")
