"""CPU tests of K/V-cache attention with a per-sequence number of new tokens (mfa_attention_forward_kvcache_varlen): NULL
handles, bad geometry and malformed host-readable cu_seqlens_q are argument errors, and without a device the call reports
MFA_ERROR_DEVICE_NOT_SUPPORTED -- never a crash, never a CPU fallback."""
import ctypes

import numpy as np
import pytest

INVALID_ARGS, DEVICE_NOT_SUPPORTED = 1, 3
BF16, FP32 = 1, 2


def _call(lib, ctx, bufs, table, *, n=2, T=5, msq=4, H=8, Hkv=2, D=64, cap=256, page=16, pages=32, in_prec=BF16,
          out_prec=FP32):
    return lib.mfa_attention_forward_kvcache_varlen(ctx, *bufs, table, n, T, msq, H, Hkv, D, cap, page, pages, 0.125, True, -1,
                                                    in_prec, out_prec, None)


def _placeholder():
    keep = np.zeros(4096, np.uint8)
    return keep, ctypes.c_void_p(keep.ctypes.data)


def test_kvcache_varlen_null_handles_are_invalid_args():
    from umfa import _ffi
    lib = _ffi._lib
    keep, h = _placeholder()
    assert _call(lib, None, [None] * 7, None) == INVALID_ARGS
    for i in (0, 1, 2, 3, 5, 6):                   # q, k_cache, v_cache, out, cu_seqlens_q, cache_seqlens (lse is optional)
        bufs = [h] * 7
        bufs[i] = None
        assert _call(lib, h, bufs, h) == INVALID_ARGS, i
    assert _call(lib, h, [h] * 7, None) == INVALID_ARGS                     # paged without a block table
    assert _call(lib, h, [h] * 7, h, page=0, pages=0) == INVALID_ARGS       # contiguous with a block table


@pytest.mark.parametrize("kw", [
    dict(page=24),                 # page_size not a multiple of 16
    dict(cap=264),                 # capacity not a multiple of the page
    dict(H=8, Hkv=3),              # num_kv_heads does not divide num_heads
    dict(H=258, Hkv=2),            # group of 129 query heads
    dict(in_prec=FP32),            # fp32 operands
    dict(D=192),                   # head_dim above 128
    dict(D=60),                    # head_dim not a multiple of 8
    dict(cap=0, page=0, pages=0),
    dict(pages=0),
    dict(n=0),                     # no sequence
    dict(T=0),                     # no query row
    dict(msq=0),
    dict(msq=6),                   # max_seqlen_q above total_q
])
def test_kvcache_varlen_bad_geometry_is_invalid_args(kw):
    from umfa import _ffi
    lib = _ffi._lib
    keep, h = _placeholder()
    table = None if kw.get("page", 16) == 0 else h
    assert _call(lib, h, [h] * 7, table, **kw) == INVALID_ARGS


def test_kvcache_varlen_without_device_reports_it():
    import umfa
    from umfa import _ffi
    if umfa.is_metal_available():
        pytest.skip("a GPU is present")
    lib = _ffi._lib
    keep, h = _placeholder()
    assert _call(lib, h, [h] * 7, h) == DEVICE_NOT_SUPPORTED
    assert _call(lib, h, [h] * 7, None, page=0, pages=0) == DEVICE_NOT_SUPPORTED
    assert _call(lib, h, [h, h, h, h, None, h, h], h) == DEVICE_NOT_SUPPORTED       # lse is optional


def test_umfa_kvcache_varlen_argument_validation():
    from umfa import core
    q = np.zeros((7, 8, 16), np.uint16)
    kc = np.zeros((3, 64, 2, 16), np.uint16)
    dims = core._kvcache_varlen_dims(q, kc, kc, [0, 1, 1, 7], [5, 9, 20], None, None)
    assert dims[:9] == (3, 7, 6, 8, 2, 16, 64, 0, 0)
    assert core._kvcache_varlen_dims(q, kc, kc, [0, 1, 1, 7], [5, 9, 20], None, 8)[2] == 8
    pool = np.zeros((10, 16, 2, 16), np.uint16)
    table = np.zeros((3, 4), np.int32)
    assert core._kvcache_varlen_dims(q, pool, pool, [0, 1, 1, 7], [5, 9, 20], table, None)[:9] == (3, 7, 6, 8, 2, 16, 64, 16, 10)
    for cu, msq in (([1, 1, 1, 7], None),          # does not start at 0
                    ([0, 3, 1, 7], None),          # decreases
                    ([0, 1, 1, 6], None),          # does not end at total_q
                    ([0, 1, 1, 7], 5)):            # a segment longer than max_seqlen_q
        with pytest.raises(ValueError):
            core._kvcache_varlen_dims(q, kc, kc, cu, [5, 9, 20], None, msq)
    with pytest.raises(ValueError):
        core._kvcache_varlen_dims(q[None], kc, kc, [0, 1, 1, 7], [5, 9, 20], None, None)       # q is [total_q, H, D]
    with pytest.raises(ValueError):
        core._kvcache_varlen_dims(q, kc, kc, [7], [5, 9, 20], None, None)                      # num_seqs + 1 offsets
    with pytest.raises(ValueError):
        core._kvcache_varlen_dims(q, kc, kc, [0, 1, 7], [5, 9, 20], None, None)                # one length per sequence
    with pytest.raises(ValueError):
        core._kvcache_varlen_dims(q, kc[:2], kc[:2], [0, 1, 1, 7], [5, 9, 20], None, None)     # contiguous caches carry the batch
    with pytest.raises(ValueError):
        core._kvcache_varlen_dims(q, pool, pool, [0, 1, 1, 7], [5, 9, 20], table[:2], None)    # one block-table row per sequence
    with pytest.raises(ValueError):
        core._kvcache_varlen_dims(q, np.zeros((3, 64, 3, 16), np.uint16), np.zeros((3, 64, 3, 16), np.uint16), [0, 1, 1, 7],
                                  [5, 9, 20], None, None)                                      # Hkv does not divide H


def test_torch_kvcache_varlen_adapter_argument_errors():
    torch = pytest.importorskip("torch")
    from pytorch_custom_op_ffi import metal_flash_attention_varlen_with_kvcache as f
    q = torch.zeros(5, 4, 64, dtype=torch.bfloat16)
    kc = torch.zeros(2, 128, 1, 64, dtype=torch.bfloat16)
    cu = torch.tensor([0, 1, 5], dtype=torch.int32)
    lens = torch.tensor([4, 9], dtype=torch.int32)
    with pytest.raises(RuntimeError, match="CUDA"):
        f(q, kc, kc, cu, lens, 4)
    with pytest.raises(RuntimeError, match="no backward"):
        f(q.clone().requires_grad_(), kc, kc, cu, lens, 4)
    with pytest.raises(RuntimeError, match="max_seqlen_q"):
        f(q, kc, kc, cu, lens, None)
    with pytest.raises(RuntimeError, match="max_seqlen_q"):
        f(q, kc, kc, cu, lens, torch.tensor(4))
