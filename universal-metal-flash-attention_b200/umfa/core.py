"""High-level numpy API over libMFAFFI.so -- host-side mirror of the reference's
examples/python-ffi/src/umfa/core.py (same class / function names, argument meaning and error behaviour),
extended with the pieces the reference only reaches through its PyTorch adapter (LSE, backward, runtime
quantisation, sliding window).

Array layout: 2-D [seq, head_dim] (single head) or 4-D.  4-D arrays are [batch, seq, heads, head_dim]
("bshd", what the reference docstrings say, core.py:286-288 there) unless layout="bhsd" is passed; bshd
arrays with heads > 1 are handed to the library through BHSD element strides, not copied.
"""
import ctypes
import weakref
from typing import NamedTuple, Optional, Tuple, Union

import numpy as np

from ._ffi import (MFA_MASK_SCALAR_BF16, MFA_MASK_SCALAR_BYTE, MFA_MASK_SCALAR_FP16, MFA_MASK_SCALAR_FP32,
                   MFA_MASK_TYPE_ADDITIVE, MFA_MASK_TYPE_BOOL, MFA_MASK_TYPE_NONE, MFA_PRECISION_BF16,
                   MFA_PRECISION_FP16, MFA_PRECISION_FP32, MFA_PRECISION_INT4, MFA_PRECISION_INT8, MFAError,
                   _check_error, _lib, mfa_buffer_t, mfa_context_t)

Precision = Union[int, str]

_PRECISIONS = {
    "fp16": MFA_PRECISION_FP16, "half": MFA_PRECISION_FP16, "float16": MFA_PRECISION_FP16,
    "bf16": MFA_PRECISION_BF16, "bfloat16": MFA_PRECISION_BF16,
    "fp32": MFA_PRECISION_FP32, "float": MFA_PRECISION_FP32, "float32": MFA_PRECISION_FP32,
    "int8": MFA_PRECISION_INT8, "int4": MFA_PRECISION_INT4,
}
_ITEMSIZE = {MFA_PRECISION_FP16: 2, MFA_PRECISION_BF16: 2, MFA_PRECISION_FP32: 4, MFA_PRECISION_INT8: 1}


def _parse_precision(precision: Precision) -> int:
    if isinstance(precision, (int, np.integer)):
        return int(precision)
    key = str(precision).lower()
    if key not in _PRECISIONS:
        raise ValueError(f"Unknown precision: {precision}. Use one of {sorted(_PRECISIONS)}")
    return _PRECISIONS[key]


class MFAContext:
    """Owns one reference on the library's device context; usable as a context manager."""

    def __init__(self):
        self._handle = mfa_context_t()
        _check_error(_lib.mfa_create_context(ctypes.byref(self._handle)))
        self._finalizer = weakref.finalize(self, MFAContext._cleanup, self._handle)

    def __enter__(self) -> "MFAContext":
        return self

    def __exit__(self, exc_type, exc, tb):
        self.close()

    def close(self):
        if self._finalizer.detach():
            MFAContext._cleanup(self._handle)

    @staticmethod
    def _cleanup(handle):
        if handle:
            _lib.mfa_destroy_context(handle)

    @property
    def handle(self):
        return self._handle

    @property
    def gpu_latency(self) -> float:
        """Device time in seconds of the last blocking operation (mfa_get_gpu_latency)."""
        return float(_lib.mfa_get_gpu_latency(self._handle))

    @property
    def last_kernel(self) -> str:
        return _lib.mfa_last_kernel_name(self._handle).decode()

    @property
    def launch_count(self) -> int:
        return int(_lib.mfa_launch_count(self._handle))

    def __bool__(self) -> bool:
        return bool(self._handle)


class MFABuffer:
    """Library view of caller memory (numpy array: wrapped, never copied on the host side) or a fresh allocation.

    strides: optional BHSD element strides (with `shape`) for non-BHSD-contiguous 4-D operands.
    device_ptr: wrap a raw CUDA device pointer (e.g. torch.Tensor.data_ptr()) of `size` bytes.
    """

    def __init__(self, context: MFAContext, data: Optional[np.ndarray] = None, size: Optional[int] = None, *,
                 shape=None, strides=None, device_ptr: Optional[int] = None):
        self._context = context
        self._handle = mfa_buffer_t()
        self._array = data
        meta = None
        if shape is not None and strides is not None:
            n = len(shape)
            meta = ((ctypes.c_int64 * n)(*[int(s) for s in shape]), (ctypes.c_int64 * n)(*[int(s) for s in strides]), n)
        if device_ptr is not None:
            if size is None:
                raise ValueError("device_ptr needs size (bytes)")
            if meta:
                rc = _lib.mfa_buffer_from_mtl_buffer_with_strides(context.handle, ctypes.c_void_p(device_ptr), size,
                                                                  meta[0], meta[1], meta[2], ctypes.byref(self._handle))
            else:
                rc = _lib.mfa_buffer_from_mtl_buffer(context.handle, ctypes.c_void_p(device_ptr), size,
                                                     ctypes.byref(self._handle))
            _check_error(rc)
        elif data is not None:
            if not data.flags.c_contiguous:
                raise ValueError("Array must be C-contiguous for zero-copy")
            ptr = data.ctypes.data_as(ctypes.c_void_p)
            if data.nbytes == 0:
                ptr = ctypes.c_void_p(ctypes.addressof(ctypes.c_char()))   # a valid non-NULL address for empty arrays
                self._keep = ptr
            if meta:
                rc = _lib.mfa_buffer_from_ptr_with_strides(context.handle, ptr, data.nbytes, meta[0], meta[1], meta[2],
                                                           ctypes.byref(self._handle))
            else:
                rc = _lib.mfa_buffer_from_ptr(context.handle, ptr, data.nbytes, ctypes.byref(self._handle))
            _check_error(rc)
        elif size is not None:
            _check_error(_lib.mfa_create_buffer(context.handle, size, ctypes.byref(self._handle)))
        else:
            raise ValueError("Must provide either data array or buffer size")
        self._finalizer = weakref.finalize(self, MFABuffer._cleanup, self._handle)

    def close(self):
        if self._finalizer.detach():
            MFABuffer._cleanup(self._handle)

    @staticmethod
    def _cleanup(handle):
        if handle:
            _lib.mfa_destroy_buffer(handle)

    @property
    def handle(self):
        return self._handle

    def contents_ptr(self):
        return _lib.mfa_buffer_contents(self._handle)

    def __bool__(self) -> bool:
        return bool(self._handle)


try:
    _BF16_DTYPE = np.dtype("bfloat16")
except TypeError:
    _BF16_DTYPE = None


class _MaskMetadata(NamedTuple):
    array: np.ndarray
    ptr: ctypes.c_void_p
    size_bytes: int
    shape: ctypes.Array
    strides: ctypes.Array
    ndim: int
    mask_type: int
    mask_scalar: int


_NO_MASK = (None, 0, None, None, 0, MFA_MASK_TYPE_NONE, MFA_MASK_SCALAR_BYTE)


def _prepare_mask_metadata(mask, bhqk: Tuple[int, int, int, int], mask_precision: Optional[Precision] = None):
    """Mask -> FFI metadata.  bool / integer arrays are BOOL masks where non-zero = attend (the kernel's rule,
    MFABridge.swift:201-205); float arrays are additive.  The mask keeps its own (broadcastable) shape -- the
    library broadcasts right-aligned against [B,H,Sq,Skv] -- so nothing is materialised on the host.
    uint16 arrays with mask_precision="bf16" carry bf16 bit patterns."""
    m = np.asarray(mask)
    mtype, mscalar = MFA_MASK_TYPE_ADDITIVE, MFA_MASK_SCALAR_FP32
    if mask_precision is not None and _parse_precision(mask_precision) == MFA_PRECISION_BF16:
        mscalar = MFA_MASK_SCALAR_BF16
        m = m.view(np.uint16) if m.dtype.itemsize == 2 else m
    elif m.dtype == np.bool_ or m.dtype in (np.int8, np.uint8, np.int16, np.uint16):
        mtype, mscalar = MFA_MASK_TYPE_BOOL, MFA_MASK_SCALAR_BYTE
        m = (m != 0).astype(np.uint8)
    elif m.dtype == np.float16:
        mscalar = MFA_MASK_SCALAR_FP16
    elif _BF16_DTYPE is not None and m.dtype == _BF16_DTYPE:
        mscalar = MFA_MASK_SCALAR_BF16
    elif m.dtype == np.float32:
        pass
    elif m.dtype == np.float64:
        m = m.astype(np.float32)
    else:
        raise ValueError("Unsupported attention mask dtype. Use bool for binary masks or "
                         "float16/bfloat16/float32 values for additive masks.")
    if m.ndim > 4:
        raise ValueError("Attention mask may have at most 4 dimensions")
    try:
        np.broadcast_shapes(m.shape, bhqk)
    except ValueError as exc:
        raise ValueError(f"Attention mask with shape {m.shape} cannot broadcast to {bhqk}.") from exc
    if np.broadcast_shapes(m.shape, bhqk) != tuple(bhqk):
        raise ValueError(f"Attention mask with shape {m.shape} cannot broadcast to {bhqk}.")
    m = np.ascontiguousarray(m)
    shape = (ctypes.c_int64 * max(m.ndim, 1))(*m.shape)
    strides = (ctypes.c_int64 * max(m.ndim, 1))(*[s // m.itemsize for s in m.strides])
    return _MaskMetadata(m, ctypes.c_void_p(m.ctypes.data), m.nbytes, shape, strides, m.ndim, mtype, mscalar)


def _mask_args(meta):
    if meta is None:
        return _NO_MASK
    return (meta.ptr, meta.size_bytes, meta.shape, meta.strides, meta.ndim, meta.mask_type, meta.mask_scalar)


class _Dims(NamedTuple):
    B: int
    H: int
    Sq: int
    Skv: int
    D: int
    bshd: bool


def _dims(q, k, v, layout: str) -> _Dims:
    if not all(isinstance(x, np.ndarray) for x in (q, k, v)):
        raise TypeError("q, k, v must be numpy arrays")
    if q.ndim == 2:
        Sq, D = q.shape
        Skv = k.shape[0]
        if k.shape != (Skv, D) or v.shape != (Skv, D):
            raise ValueError(f"Shape mismatch: q={q.shape}, k={k.shape}, v={v.shape}")
        return _Dims(1, 1, Sq, Skv, D, False)
    if q.ndim == 4:
        if layout == "bshd":
            B, Sq, H, D = q.shape
            Skv = k.shape[1]
            want = (B, Skv, H, D)
        elif layout == "bhsd":
            B, H, Sq, D = q.shape
            Skv = k.shape[2]
            want = (B, H, Skv, D)
        else:
            raise ValueError("layout must be 'bshd' or 'bhsd'")
        if k.shape != want or v.shape != want:
            raise ValueError(f"Shape mismatch: q={q.shape}, k={k.shape}, v={v.shape}")
        return _Dims(B, H, Sq, Skv, D, layout == "bshd" and H > 1)
    raise ValueError(f"Invalid tensor dimensions. Expected 2D or 4D, got q.shape={q.shape}")


def _operand(ctx, arr, d: _Dims, S: int):
    """Wrap one [.., S, .., D] operand; bshd arrays with several heads travel as BHSD strides."""
    if d.bshd:
        return MFABuffer(ctx, arr, shape=(d.B, d.H, S, d.D), strides=(S * d.H * d.D, d.D, d.H * d.D, 1))
    return MFABuffer(ctx, arr)


def _np_dtype_for(prec: int):
    return {MFA_PRECISION_FP16: np.float16, MFA_PRECISION_FP32: np.float32}.get(prec)


def _check_input_dtype(x: np.ndarray, prec: int, name: str):
    if x.dtype.itemsize != _ITEMSIZE.get(prec, x.dtype.itemsize):
        raise ValueError(f"{name} has dtype {x.dtype} but input_precision needs {_ITEMSIZE[prec]}-byte elements "
                         "(bf16 data travels as uint16 bit patterns)")


def flash_attention_forward(context: MFAContext, q, k, v, *, attn_mask=None, causal: bool = False,
                            softmax_scale: Optional[float] = None, input_precision: Precision = "fp16",
                            intermediate_precision: Precision = "fp16", output_precision: Precision = "fp16",
                            layout: str = "bshd", window_size: Optional[int] = None, return_lse: bool = False,
                            mask_precision: Optional[Precision] = None):
    """O = softmax(scale * Q K^T [+ mask]) V through mfa_attention_forward (or mfa_attention_forward_ex when a
    sliding window or the LSE is requested).

    Returns an array shaped like q.  The library writes O as fp32 (the reference engine's contract); it is
    returned as fp32 unless q is float16 and output_precision is fp16, in which case the library writes fp16
    directly into a q-shaped array -- the reference adapter's behaviour (core.py:375 there).
    bf16 inputs are uint16 arrays of bit patterns with input_precision="bf16".
    With return_lse=True returns (O, L) where L = log2(e) * logsumexp(scale * S), shape [B,H,Sq] (or [Sq])."""
    d = _dims(q, k, v, layout)
    if softmax_scale is None:
        softmax_scale = 1.0 / np.sqrt(d.D)
    in_prec = _parse_precision(input_precision)
    mid_prec = _parse_precision(intermediate_precision)
    out_prec = _parse_precision(output_precision)
    for name, x in (("q", q), ("k", k), ("v", v)):
        _check_input_dtype(x, in_prec, name)
    meta = None
    if attn_mask is not None:
        meta = _prepare_mask_metadata(attn_mask, (d.B, d.H, d.Sq, d.Skv), mask_precision)
    out_dtype = np.float32
    if q.dtype == np.float16 and out_prec == MFA_PRECISION_FP16:
        out_dtype = np.float16
    if d.bshd:
        out_dtype = np.float32      # strided output path writes fp32
    output = np.zeros(q.shape, dtype=out_dtype)
    lse = np.zeros((d.B, d.H, d.Sq), np.float32) if return_lse else None
    bufs = [_operand(context, q, d, d.Sq), _operand(context, k, d, d.Skv), _operand(context, v, d, d.Skv),
            _operand(context, output, d, d.Sq)]
    if lse is not None:
        bufs.append(MFABuffer(context, lse))
    try:
        if window_size is None and lse is None:
            rc = _lib.mfa_attention_forward(
                context.handle, bufs[0].handle, bufs[1].handle, bufs[2].handle, bufs[3].handle,
                d.B, d.Sq, d.Skv, d.H, d.D, softmax_scale, causal, in_prec, mid_prec,
                out_prec if out_dtype != np.float32 else MFA_PRECISION_FP32, False, False, False, False,
                *_mask_args(meta))
        else:
            rc = _lib.mfa_attention_forward_ex(
                context.handle, bufs[0].handle, bufs[1].handle, bufs[2].handle, bufs[3].handle,
                bufs[4].handle if lse is not None else None, d.B, d.Sq, d.Skv, d.H, d.D, softmax_scale, causal,
                -1 if window_size is None else int(window_size), in_prec,
                out_prec if out_dtype != np.float32 else MFA_PRECISION_FP32, *_mask_args(meta), None)
        _check_error(rc)
    finally:
        for b in bufs:
            b.close()
    if return_lse:
        return output, (lse.reshape(d.Sq) if q.ndim == 2 else lse)
    return output


def flash_attention_backward(context: MFAContext, d_out, q, k, v, out, lse, *, attn_mask=None, causal: bool = False,
                             softmax_scale: Optional[float] = None, input_precision: Precision = "fp32",
                             layout: str = "bhsd", window_size: Optional[int] = None,
                             mask_precision: Optional[Precision] = None):
    """dQ, dK, dV (fp32) and D through mfa_attention_backward / mfa_attention_backward_ex.
    d_out, q, k, v share input_precision; out is the forward's fp32 O; lse its L (log2 units).
    Only contiguous BHSD (or 2-D) operands.  Returns (dq, dk, dv, dterm)."""
    if layout != "bhsd" and q.ndim == 4:
        raise ValueError("backward takes layout='bhsd'")
    d = _dims(q, k, v, "bhsd")
    if softmax_scale is None:
        softmax_scale = 1.0 / np.sqrt(d.D)
    in_prec = _parse_precision(input_precision)
    for name, x in (("q", q), ("k", k), ("v", v), ("d_out", d_out)):
        _check_input_dtype(x, in_prec, name)
    out = np.ascontiguousarray(out, np.float32)
    lse = np.ascontiguousarray(lse, np.float32)
    meta = None
    if attn_mask is not None:
        meta = _prepare_mask_metadata(attn_mask, (d.B, d.H, d.Sq, d.Skv), mask_precision)
    dq = np.zeros(q.shape, np.float32)
    dk = np.zeros(k.shape, np.float32)
    dv = np.zeros(v.shape, np.float32)
    dterm = np.zeros((d.B, d.H, d.Sq), np.float32)
    arrays = [np.ascontiguousarray(d_out), q, k, v, out, lse, dq, dk, dv, dterm]
    bufs = [MFABuffer(context, a) for a in arrays]
    h = [b.handle for b in bufs]
    try:
        if window_size is None and meta is None:
            rc = _lib.mfa_attention_backward(context.handle, *h, d.B, d.Sq, d.Skv, d.H, d.D, softmax_scale, causal,
                                             in_prec, MFA_PRECISION_FP32, False, False, False, False)
        else:
            rc = _lib.mfa_attention_backward_ex(context.handle, *h, d.B, d.Sq, d.Skv, d.H, d.D, softmax_scale, causal,
                                                -1 if window_size is None else int(window_size), in_prec,
                                                *_mask_args(meta), None)
        _check_error(rc)
    finally:
        for b in bufs:
            b.close()
    return dq, dk, dv, (dterm.reshape(d.Sq) if q.ndim == 2 else dterm)


def _varlen_dims(q, k, v, cu_seqlens_q, cu_seqlens_k, layout: str):
    """(H, Hkv, total_q, total_k, D, cu_q, cu_k) of packed [total, heads, D] ("thd") or [heads, total, D] ("hsd") operands."""
    if not all(isinstance(x, np.ndarray) and x.ndim == 3 for x in (q, k, v)):
        raise ValueError("varlen q, k, v must be 3-D numpy arrays")
    if layout == "thd":
        (Tq, H, D), (Tk, Hkv, Dk) = q.shape, k.shape
    elif layout == "hsd":
        (H, Tq, D), (Hkv, Tk, Dk) = q.shape, k.shape
    else:
        raise ValueError("layout must be 'thd' or 'hsd'")
    if v.shape != k.shape or Dk != D or Hkv == 0 or H % Hkv:
        raise ValueError(f"Shape mismatch: q={q.shape}, k={k.shape}, v={v.shape}")
    cu_q = np.ascontiguousarray(cu_seqlens_q, np.int32)
    cu_k = np.ascontiguousarray(cu_seqlens_k, np.int32)
    if cu_q.ndim != 1 or cu_q.shape != cu_k.shape or cu_q.size < 2:
        raise ValueError("cu_seqlens_q / cu_seqlens_k must be 1-D int32 arrays of num_seqs + 1 offsets")
    return H, Hkv, Tq, Tk, D, cu_q, cu_k


def _varlen_operand(ctx, arr, heads: int, total: int, D: int, layout: str):
    """[total, heads, D] arrays travel as [1, heads, total, D] element strides; [heads, total, D] as they are."""
    if layout == "thd":
        return MFABuffer(ctx, arr, shape=(1, heads, total, D), strides=(total * heads * D, D, heads * D, 1))
    return MFABuffer(ctx, arr)


def flash_attention_varlen_forward(context: MFAContext, q, k, v, cu_seqlens_q, cu_seqlens_k, *, causal: bool = False,
                                   softmax_scale: Optional[float] = None, input_precision: Precision = "fp16",
                                   window_size: Optional[int] = None, layout: str = "thd"):
    """Attention over sequences packed along the token axis (mfa_attention_forward_varlen): segment s holds query rows
    cu_seqlens_q[s]:cu_seqlens_q[s+1] and keys cu_seqlens_k[s]:cu_seqlens_k[s+1]; a row sees only its own segment's keys, causal /
    window_size apply inside the segment (top-left aligned).  q is [total_q, H, D], k / v [total_k, Hkv, D] (layout="hsd":
    [H, total, D]); Hkv divides H (grouped-query attention).  bf16 inputs are uint16 bit patterns with input_precision="bf16".
    Returns (O fp32 shaped like q, L fp32 [H, total_q] in log2 units; rows that see no key: O = 0, L = -inf)."""
    H, Hkv, Tq, Tk, D, cu_q, cu_k = _varlen_dims(q, k, v, cu_seqlens_q, cu_seqlens_k, layout)
    if softmax_scale is None:
        softmax_scale = 1.0 / np.sqrt(D)
    in_prec = _parse_precision(input_precision)
    for name, x in (("q", q), ("k", k), ("v", v)):
        _check_input_dtype(x, in_prec, name)
    out = np.zeros(q.shape, np.float32)
    lse = np.zeros((H, Tq), np.float32)
    bufs = [_varlen_operand(context, np.ascontiguousarray(q), H, Tq, D, layout),
            _varlen_operand(context, np.ascontiguousarray(k), Hkv, Tk, D, layout),
            _varlen_operand(context, np.ascontiguousarray(v), Hkv, Tk, D, layout),
            _varlen_operand(context, out, H, Tq, D, layout), MFABuffer(context, lse),
            MFABuffer(context, cu_q), MFABuffer(context, cu_k)]
    try:
        _check_error(_lib.mfa_attention_forward_varlen(
            context.handle, *[b.handle for b in bufs], cu_q.size - 1, Tq, Tk, H, Hkv, D, softmax_scale, causal,
            -1 if window_size is None else int(window_size), in_prec, MFA_PRECISION_FP32, None))
    finally:
        for b in bufs:
            b.close()
    return out, lse


def _kvcache_dims(q, k_cache, v_cache, cache_seqlens, block_table):
    """(B, Sq, H, Hkv, D, capacity, page_size, num_pages, lens, table) of a K/V-cache call: q [B, Sq, H, D]; caches
    [B, capacity, Hkv, D] (block_table None) or paged pools [num_pages, page_size, Hkv, D] with block_table [B, pages per seq]."""
    if not all(isinstance(x, np.ndarray) and x.ndim == 4 for x in (q, k_cache, v_cache)):
        raise ValueError("kvcache q, k_cache, v_cache must be 4-D numpy arrays")
    B, Sq, H, D = q.shape
    if v_cache.shape != k_cache.shape or k_cache.shape[3] != D or k_cache.shape[2] == 0 or H % k_cache.shape[2]:
        raise ValueError(f"Shape mismatch: q={q.shape}, k_cache={k_cache.shape}, v_cache={v_cache.shape}")
    Hkv = k_cache.shape[2]
    lens = np.ascontiguousarray(cache_seqlens, np.int32)
    if lens.shape != (B,):
        raise ValueError(f"cache_seqlens must hold one length per sequence ({B}), got shape {lens.shape}")
    if block_table is None:
        if k_cache.shape[0] != B:
            raise ValueError(f"contiguous caches need batch {B}, got {k_cache.shape[0]}")
        return B, Sq, H, Hkv, D, k_cache.shape[1], 0, 0, lens, None
    table = np.ascontiguousarray(block_table, np.int32)
    if table.ndim != 2 or table.shape[0] != B:
        raise ValueError(f"block_table must be [batch, pages per sequence], got shape {table.shape}")
    num_pages, page_size = k_cache.shape[0], k_cache.shape[1]
    return B, Sq, H, Hkv, D, table.shape[1] * page_size, page_size, num_pages, lens, table


def flash_attention_kvcache(context: MFAContext, q, k_cache, v_cache, cache_seqlens, block_table=None, *,
                            causal: bool = True, window_size: Optional[int] = None, softmax_scale: Optional[float] = None,
                            input_precision: Precision = "bf16", output_precision: Precision = "fp32"):
    """Attention of Sq new tokens per sequence against that sequence's K/V cache (mfa_attention_forward_kvcache).  q is
    [B, Sq, H, D]; k_cache / v_cache are [B, capacity, Hkv, D], or with block_table ([B, capacity / page_size] int32 page ids)
    paged pools [num_pages, page_size, Hkv, D].  cache_seqlens[b] = valid keys of sequence b, the Sq new tokens included; token s
    sits at position cache_seqlens[b] - Sq + s (causal / window_size are bottom-right aligned).  bf16 data travels as uint16 bit
    patterns.  Returns (O [B, Sq, H, D] in output_precision (fp32, or fp16 / uint16 bf16 bits), L fp32 [B, H, Sq] in log2
    units); rows that see no key get O = 0, L = -inf.  Cache rows past cache_seqlens[b] inside the last 128-key tile are read
    and enter P V with weight 0, so they must hold finite values (zero-initialised caches do)."""
    B, Sq, H, Hkv, D, cap, page, npages, lens, table = _kvcache_dims(q, k_cache, v_cache, cache_seqlens, block_table)
    if softmax_scale is None:
        softmax_scale = 1.0 / np.sqrt(D)
    in_prec, out_prec = _parse_precision(input_precision), _parse_precision(output_precision)
    for name, x in (("q", q), ("k_cache", k_cache), ("v_cache", v_cache)):
        _check_input_dtype(x, in_prec, name)
    out = np.zeros(q.shape, {MFA_PRECISION_FP32: np.float32, MFA_PRECISION_FP16: np.float16}.get(out_prec, np.uint16))
    lse = np.zeros((B, H, Sq), np.float32)
    bshd = lambda arr, S, Hn: MFABuffer(context, arr, shape=(B, Hn, S, D), strides=(S * Hn * D, D, Hn * D, 1))
    bufs = [bshd(np.ascontiguousarray(q), Sq, H)]
    if table is None:
        bufs += [bshd(np.ascontiguousarray(k_cache), cap, Hkv), bshd(np.ascontiguousarray(v_cache), cap, Hkv)]
    else:
        bufs += [MFABuffer(context, np.ascontiguousarray(k_cache)), MFABuffer(context, np.ascontiguousarray(v_cache))]
    bufs += [bshd(out, Sq, H), MFABuffer(context, lse), MFABuffer(context, lens)]
    if table is not None:
        bufs.append(MFABuffer(context, table))
    h = [b.handle for b in bufs]
    try:
        _check_error(_lib.mfa_attention_forward_kvcache(
            context.handle, *h[:6], h[6] if table is not None else None, B, Sq, H, Hkv, D, cap, page, npages, softmax_scale,
            causal, -1 if window_size is None else int(window_size), in_prec, out_prec, None))
    finally:
        for b in bufs:
            b.close()
    return out, lse


def flash_attention_varlen_backward(context: MFAContext, d_out, q, k, v, out, lse, cu_seqlens_q, cu_seqlens_k, *,
                                    causal: bool = False, softmax_scale: Optional[float] = None,
                                    input_precision: Precision = "fp32", window_size: Optional[int] = None,
                                    layout: str = "thd"):
    """dQ, dK, dV (fp32, shaped like q / k / v) and D ([H, total_q]) of flash_attention_varlen_forward
    (mfa_attention_backward_varlen).  d_out, q, k, v share input_precision; out / lse are the forward's fp32 results.
    With Hkv < H, dK / dV hold the sums over each group of query heads."""
    H, Hkv, Tq, Tk, D, cu_q, cu_k = _varlen_dims(q, k, v, cu_seqlens_q, cu_seqlens_k, layout)
    if softmax_scale is None:
        softmax_scale = 1.0 / np.sqrt(D)
    in_prec = _parse_precision(input_precision)
    for name, x in (("q", q), ("k", k), ("v", v), ("d_out", d_out)):
        _check_input_dtype(x, in_prec, name)
    hsd = (lambda x: np.ascontiguousarray(x.transpose(1, 0, 2))) if layout == "thd" else np.ascontiguousarray
    dq = np.zeros((H, Tq, D), np.float32)
    dk = np.zeros((Hkv, Tk, D), np.float32)
    dv = np.zeros((Hkv, Tk, D), np.float32)
    dterm = np.zeros((H, Tq), np.float32)
    bufs = [MFABuffer(context, hsd(d_out)),
            _varlen_operand(context, np.ascontiguousarray(q), H, Tq, D, layout),
            _varlen_operand(context, np.ascontiguousarray(k), Hkv, Tk, D, layout),
            _varlen_operand(context, np.ascontiguousarray(v), Hkv, Tk, D, layout),
            MFABuffer(context, hsd(np.asarray(out, np.float32))), MFABuffer(context, np.ascontiguousarray(lse, np.float32)),
            MFABuffer(context, dq), MFABuffer(context, dk), MFABuffer(context, dv), MFABuffer(context, dterm),
            MFABuffer(context, cu_q), MFABuffer(context, cu_k)]
    try:
        _check_error(_lib.mfa_attention_backward_varlen(
            context.handle, *[b.handle for b in bufs], cu_q.size - 1, Tq, Tk, H, Hkv, D, softmax_scale, causal,
            -1 if window_size is None else int(window_size), in_prec, None))
    finally:
        for b in bufs:
            b.close()
    if layout == "thd":
        dq, dk, dv = (np.ascontiguousarray(x.transpose(1, 0, 2)) for x in (dq, dk, dv))
    return dq, dk, dv, dterm


def attention(q, k, v, context: Optional[MFAContext] = None, **kwargs):
    """flash_attention_forward with automatic context management."""
    if context is not None:
        return flash_attention_forward(context, q, k, v, **kwargs)
    with MFAContext() as ctx:
        return flash_attention_forward(ctx, q, k, v, **kwargs)


def quantized_attention(q, k, v, context: Optional[MFAContext] = None, *, causal: bool = False,
                        softmax_scale: Optional[float] = None, query_precision: Precision = "bf16",
                        kv_precision: Precision = "int8", output_precision: Precision = "bf16",
                        q_scale: float = 1.0, q_zero_point: int = 0, k_scale: float = 1.0, k_zero_point: int = 0,
                        v_scale: float = 1.0, v_zero_point: int = 0):
    """mfa_attention_forward_quantized on 2-D operands: q in query_precision, k/v holding kv_precision codes with
    per-tensor scale / zero point (the reference adapter's contract, core.py:456-497 there).  Returns fp32 O."""
    if context is None:
        with MFAContext() as ctx:
            return quantized_attention(q, k, v, ctx, causal=causal, softmax_scale=softmax_scale,
                                       query_precision=query_precision, kv_precision=kv_precision,
                                       output_precision=output_precision, q_scale=q_scale, q_zero_point=q_zero_point,
                                       k_scale=k_scale, k_zero_point=k_zero_point, v_scale=v_scale,
                                       v_zero_point=v_zero_point)
    if not all(isinstance(x, np.ndarray) for x in (q, k, v)):
        raise TypeError("q, k, v must be numpy arrays")
    if q.ndim != 2:
        raise ValueError("Quantized attention currently only supports 2D tensors")
    Sq, D = q.shape
    Skv = k.shape[0]
    q_prec, kv_prec, out_prec = (_parse_precision(p) for p in (query_precision, kv_precision, output_precision))
    if softmax_scale is None:
        softmax_scale = 1.0 / np.sqrt(D)
    output = np.zeros((Sq, D), np.float32)
    bufs = [MFABuffer(context, np.ascontiguousarray(a)) for a in (q, k, v)] + [MFABuffer(context, output)]
    try:
        _check_error(_lib.mfa_attention_forward_quantized(
            context.handle, *[b.handle for b in bufs], 1, Sq, Skv, 1, D, softmax_scale, causal,
            q_scale, q_zero_point, k_scale, k_zero_point, v_scale, v_zero_point,
            q_prec, kv_prec, kv_prec, out_prec, False, False, False, False))
    finally:
        for b in bufs:
            b.close()
    return output


def runtime_quantized_attention(context: MFAContext, q, k, v, *, target_precision: Precision = "int8",
                                quant_mode: int = 0, input_precision: Precision = "fp32", causal: bool = False,
                                softmax_scale: Optional[float] = None, mask=None):
    """mfa_quantized_forward_with_lse: quantise BHSD q, k, v on the device (quant_mode 0 = per tensor, 2 = blocks of
    64 tokens), attend, return (O fp32, L).  mask: optional dense fp32 additive [B,H,Sq,Skv]."""
    d = _dims(q, k, v, "bhsd")
    if softmax_scale is None:
        softmax_scale = 1.0 / np.sqrt(d.D)
    out = np.zeros(q.shape, np.float32)
    lse = np.zeros((d.B, d.H, d.Sq), np.float32)
    arrays = [q, k, v, out, lse]
    if mask is not None:
        arrays.append(np.ascontiguousarray(np.broadcast_to(np.asarray(mask, np.float32), (d.B, d.H, d.Sq, d.Skv))))
    bufs = [MFABuffer(context, a) for a in arrays]
    try:
        _check_error(_lib.mfa_quantized_forward_with_lse(
            context.handle, *[b.handle for b in bufs[:5]], bufs[5].handle if mask is not None else None,
            d.B, d.Sq, d.Skv, d.H, d.D, softmax_scale, causal, _parse_precision(target_precision), quant_mode,
            _parse_precision(input_precision)))
    finally:
        for b in bufs:
            b.close()
    return out, lse


def runtime_quantized_backward(context: MFAContext, q, k, v, out, grad_out, lse, *, target_precision: Precision = "int8",
                               quant_mode: int = 0, input_precision: Precision = "fp32", causal: bool = False,
                               softmax_scale: Optional[float] = None, mask=None):
    """mfa_quantized_backward: returns (dq, dk, dv) fp32."""
    d = _dims(q, k, v, "bhsd")
    if softmax_scale is None:
        softmax_scale = 1.0 / np.sqrt(d.D)
    dq, dk, dv = (np.zeros(x.shape, np.float32) for x in (q, k, v))
    arrays = [q, k, v, np.ascontiguousarray(out, np.float32), np.ascontiguousarray(grad_out, np.float32),
              np.ascontiguousarray(lse, np.float32), dq, dk, dv]
    if mask is not None:
        arrays.append(np.ascontiguousarray(np.broadcast_to(np.asarray(mask, np.float32), (d.B, d.H, d.Sq, d.Skv))))
    bufs = [MFABuffer(context, a) for a in arrays]
    try:
        _check_error(_lib.mfa_quantized_backward(
            context.handle, *[b.handle for b in bufs[:9]], bufs[9].handle if mask is not None else None,
            d.B, d.Sq, d.Skv, d.H, d.D, softmax_scale, causal, _parse_precision(target_precision), quant_mode,
            _parse_precision(input_precision)))
    finally:
        for b in bufs:
            b.close()
    return dq, dk, dv


def quantize(context: MFAContext, x: np.ndarray, *, bits: int = 8, block_rows: int = 0, block_cols: int = 0,
             src_precision: Precision = "fp32", scale_floor: float = 0.0):
    """mfa_quantize on a 2-D [rows, cols] array.  Returns (codes, scales): int8 [rows, cols] or packed uint8
    [(rows*cols+1)//2]; scales fp32 [n_blocks] (row-major over block_rows x block_cols tiles; 0 = full extent)."""
    if x.ndim != 2:
        raise ValueError("quantize takes a 2-D array")
    rows, cols = x.shape
    br = rows if block_rows in (0, None) else min(block_rows, rows)
    bc = cols if block_cols in (0, None) else min(block_cols, cols)
    nb = (-(-rows // br)) * (-(-cols // bc)) if rows and cols else 0
    n = rows * cols
    codes = np.zeros(n if bits == 8 else (n + 1) // 2, np.uint8)
    scales = np.zeros(max(nb, 1), np.float32)
    bufs = [MFABuffer(context, np.ascontiguousarray(x)), MFABuffer(context, codes), MFABuffer(context, scales)]
    try:
        _check_error(_lib.mfa_quantize(context.handle, bufs[0].handle, bufs[1].handle, bufs[2].handle, rows, cols,
                                       block_rows or 0, block_cols or 0, _parse_precision(src_precision),
                                       MFA_PRECISION_INT8 if bits == 8 else MFA_PRECISION_INT4, scale_floor, None))
    finally:
        for b in bufs:
            b.close()
    scales = scales[:nb]
    return (codes.view(np.int8).reshape(rows, cols) if bits == 8 else codes), scales
