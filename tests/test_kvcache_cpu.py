"""CPU tests of the K/V-cache attention symbol: NULL handles and bad geometry are argument errors, and without a device the call
reports MFA_ERROR_DEVICE_NOT_SUPPORTED -- never a crash, never a CPU fallback."""
import ctypes

import numpy as np
import pytest

INVALID_ARGS, DEVICE_NOT_SUPPORTED = 1, 3
BF16, FP32 = 1, 2


def _call(lib, ctx, bufs, table, *, B=2, Sq=1, H=8, Hkv=2, D=64, cap=256, page=16, pages=32, in_prec=BF16, out_prec=FP32):
    return lib.mfa_attention_forward_kvcache(ctx, *bufs, table, B, Sq, H, Hkv, D, cap, page, pages, 0.125, True, -1,
                                             in_prec, out_prec, None)


def _placeholder():
    keep = np.zeros(4096, np.uint8)
    return keep, ctypes.c_void_p(keep.ctypes.data)


def test_kvcache_null_handles_are_invalid_args():
    from umfa import _ffi
    lib = _ffi._lib
    keep, h = _placeholder()
    assert _call(lib, None, [None] * 6, None) == INVALID_ARGS
    for i in (0, 1, 2, 3, 5):                      # q, k_cache, v_cache, out, cache_seqlens (lse is optional)
        bufs = [h] * 6
        bufs[i] = None
        assert _call(lib, h, bufs, h) == INVALID_ARGS, i
    assert _call(lib, h, [h] * 6, None) == INVALID_ARGS                     # paged without a block table
    assert _call(lib, h, [h] * 6, h, page=0, pages=0) == INVALID_ARGS       # contiguous with a block table


@pytest.mark.parametrize("kw", [
    dict(page=24),                 # page_size not a multiple of 16
    dict(cap=264),                 # capacity not a multiple of the page
    dict(H=8, Hkv=3),              # num_kv_heads does not divide num_heads
    dict(H=258, Hkv=2),            # group of 129 query heads
    dict(in_prec=FP32),            # fp32 operands
    dict(D=192),                   # head_dim above 128
    dict(D=60),                    # head_dim not a multiple of 8
    dict(B=0),
    dict(Sq=0),
    dict(cap=0, page=0, pages=0),
    dict(pages=0),
])
def test_kvcache_bad_geometry_is_invalid_args(kw):
    from umfa import _ffi
    lib = _ffi._lib
    keep, h = _placeholder()
    table = None if kw.get("page", 16) == 0 else h
    assert _call(lib, h, [h] * 6, table, **kw) == INVALID_ARGS


def test_kvcache_without_device_reports_it():
    import umfa
    from umfa import _ffi
    if umfa.is_metal_available():
        pytest.skip("a GPU is present")
    lib = _ffi._lib
    keep, h = _placeholder()
    assert _call(lib, h, [h] * 6, h) == DEVICE_NOT_SUPPORTED
    assert _call(lib, h, [h] * 6, None, page=0, pages=0) == DEVICE_NOT_SUPPORTED
    assert _call(lib, h, [h, h, h, h, None, h], h) == DEVICE_NOT_SUPPORTED          # lse is optional


def test_umfa_kvcache_argument_validation():
    from umfa import core
    q = np.zeros((2, 3, 8, 16), np.uint16)
    kc = np.zeros((2, 64, 2, 16), np.uint16)
    assert core._kvcache_dims(q, kc, kc, [5, 9], None)[:8] == (2, 3, 8, 2, 16, 64, 0, 0)
    pool = np.zeros((10, 16, 2, 16), np.uint16)
    table = np.zeros((2, 4), np.int32)
    assert core._kvcache_dims(q, pool, pool, [5, 9], table)[:8] == (2, 3, 8, 2, 16, 64, 16, 10)
    with pytest.raises(ValueError):
        core._kvcache_dims(q, np.zeros((2, 64, 3, 16), np.uint16), np.zeros((2, 64, 3, 16), np.uint16), [5, 9], None)
    with pytest.raises(ValueError):
        core._kvcache_dims(q, kc, kc, [5], None)                 # one length per sequence
    with pytest.raises(ValueError):
        core._kvcache_dims(q, kc[:1], kc[:1], [5, 9], None)      # contiguous caches carry the batch
    with pytest.raises(ValueError):
        core._kvcache_dims(q, pool, pool, [5, 9], table[:1])     # one block-table row per sequence
    with pytest.raises(ValueError):
        core._kvcache_dims(q[0], kc, kc, [5, 9], None)


def test_torch_kvcache_adapter_argument_errors():
    torch = pytest.importorskip("torch")
    from pytorch_custom_op_ffi import metal_flash_attention_with_kvcache
    q = torch.zeros(1, 1, 4, 64, dtype=torch.bfloat16)
    kc = torch.zeros(1, 128, 1, 64, dtype=torch.bfloat16)
    lens = torch.tensor([4], dtype=torch.int32)
    with pytest.raises(RuntimeError, match="CUDA"):
        metal_flash_attention_with_kvcache(q, kc, kc, lens)
    with pytest.raises(RuntimeError, match="no backward"):
        metal_flash_attention_with_kvcache(q.clone().requires_grad_(), kc, kc, lens)
