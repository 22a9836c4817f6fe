"""CUDA twin of the reference's compiled torch extension `metal_sdpa_extension`
(examples/pytorch-custom-op-ffi/src/python_bindings.cpp:40-170 lists the functions; the C++ behind them is
src/metal_sdpa_backend.cpp:1643-1904 (SDPA entry and dispatch), :2672-2861 (MetalFlashAttentionFn),
:3139-3383 (quantised autograd Function), :1440-1560 (RoPE + SDPA), :3395-3420 (Hadamard)).

Same function names, argument meaning and error behaviour; the difference is what sits underneath: CUDA tensors are
handed to libMFAFFI.so zero-copy (`mfa_buffer_from_mtl_buffer(data_ptr)`), and the dense paths are enqueued on
torch's current CUDA stream through the additive `mfa_attention_{forward,backward}_ex` symbols -- no
`.contiguous()` round trip through the CPU, no host synchronisation.  The quantised entry points are the
reference's blocking `mfa_quantized_forward_with_lse` / `mfa_quantized_backward`.

There is no eager / PyTorch fallback in this module: unsupported inputs raise.  (backend.py decides whether a call to
F.scaled_dot_product_attention is routed here at all.)
"""
import ctypes
import math
import threading
from typing import Optional

import torch

from umfa import _ffi
from umfa.core import MFAContext

_lib = _ffi._lib

QUANT_NONE = 0
QUANT_INT8 = 3           # MetalSDPABackend::QUANT_INT8 (= MFA_PRECISION_INT8)
QUANT_INT4 = 4
QUANT_TENSOR_WISE = 0
QUANT_BLOCK_WISE = 2

_PREC = {torch.float16: _ffi.MFA_PRECISION_FP16, torch.bfloat16: _ffi.MFA_PRECISION_BF16,
         torch.float32: _ffi.MFA_PRECISION_FP32}
_MASK_SCALAR = {torch.float16: _ffi.MFA_MASK_SCALAR_FP16, torch.bfloat16: _ffi.MFA_MASK_SCALAR_BF16,
                torch.float32: _ffi.MFA_MASK_SCALAR_FP32}

_state = threading.local()
_lock = threading.Lock()
_ctx: Optional[MFAContext] = None            # the first context created (kept for introspection in tests)
_ctxs = {}                                   # device index -> context
_quant = {"precision": QUANT_NONE, "block_mode": QUANT_TENSOR_WISE}
_STAT_KEYS = ("total", "quantized_autograd", "fp32_autograd", "direct", "mask_all_true_skipped", "fallback_native")
_stats = {k: 0 for k in _STAT_KEYS}


def _context(device: torch.device) -> MFAContext:
    """One retained library context per CUDA device (mfa_set_device selects the device of the next mfa_create_context), so
    tensors on any GPU of the process are served by the context that lives on their device."""
    global _ctx
    idx = device.index if device.index is not None else torch.cuda.current_device()
    with _lock:
        ctx = _ctxs.get(idx)
        if ctx is None:
            rc = _lib.mfa_set_device(idx)
            if rc != 0:
                raise RuntimeError(f"mfa_set_device({idx}) failed with code {rc}")
            ctx = MFAContext()
            ctx.device_index = idx
            _ctxs[idx] = ctx
            if _ctx is None:
                _ctx = ctx
        return ctx


def device_supported(device: torch.device) -> bool:
    """True when `device` is a GPU libMFAFFI.so has kernels for (compute capability 10.x)."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    try:
        return torch.cuda.get_device_capability(idx)[0] == 10
    except Exception:
        return False


class _Bound:
    """mfa_buffer_t views over CUDA tensors for the duration of one call."""

    def __init__(self, ctx):
        self.ctx, self.handles = ctx, []

    def __call__(self, t: Optional[torch.Tensor]):
        if t is None:
            return None
        h = _ffi.mfa_buffer_t()
        nbytes = max(t.numel() * t.element_size(), 1)
        _ffi._check_error(_lib.mfa_buffer_from_mtl_buffer(self.ctx.handle, ctypes.c_void_p(t.data_ptr()), nbytes,
                                                          ctypes.byref(h)))
        self.handles.append(h)
        return h

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        for h in self.handles:
            _lib.mfa_destroy_buffer(h)


def _check_inputs(query, key, value):
    if not (query.is_cuda and key.is_cuda and value.is_cuda):
        raise RuntimeError("Metal SDPA Backend Error: tensors must live on a CUDA device (B200 build)")
    if query.dim() != 4 or key.dim() != 4 or value.dim() != 4:
        raise RuntimeError("Unsupported tensor dimensions. Expected 4D (batch, num_heads, seq_len, head_dim)")
    if query.dtype not in _PREC:
        raise RuntimeError("Unsupported dtype for Metal Flash Attention. Supported: float16, float32, bfloat16")
    if key.dtype != query.dtype or value.dtype != query.dtype:
        raise RuntimeError("Query, key, and value tensors must have the same dtype")
    if key.size(2) != value.size(2):
        raise RuntimeError("Metal SDPA: key and value must have matching sequence lengths")
    if query.size(3) > 256:
        raise RuntimeError("Head dimension too large (max 256)")


def _expand_gqa(query, key, value):
    """GQA: repeat each KV head Hq/Hkv times (metal_sdpa_backend.cpp:1703-1712)."""
    hq, hkv = query.size(1), key.size(1)
    if hq != hkv:
        if hq > hkv and hq % hkv == 0:
            g = hq // hkv
            key, value = key.repeat_interleave(g, 1), value.repeat_interleave(g, 1)
        else:
            raise RuntimeError(f"Metal SDPA: {hq} query heads are not a multiple of {hkv} key/value heads")
    return key, value


def _mask_args(mask: Optional[torch.Tensor], query, keep):
    """-> the seven C mask arguments.  bool: True = attend (MFABridge.swift:201-205); additive masks keep PyTorch
    semantics softmax(scale*QK^T + mask) (SURVEY quirk Q7)."""
    if mask is None:
        return [None, 0, None, None, 0, _ffi.MFA_MASK_TYPE_NONE, _ffi.MFA_MASK_SCALAR_BYTE]
    if mask.dim() == 0 or mask.dim() > 4:
        raise RuntimeError("Unsupported attn_mask rank for Metal Flash Attention (1..4 dims)")
    if mask.device != query.device:
        mask = mask.to(query.device)
    if mask.dtype == torch.bool:
        mtype, scalar = _ffi.MFA_MASK_TYPE_BOOL, _ffi.MFA_MASK_SCALAR_BYTE
    elif mask.dtype in _MASK_SCALAR:
        mtype, scalar = _ffi.MFA_MASK_TYPE_ADDITIVE, _MASK_SCALAR[mask.dtype]
    else:
        raise RuntimeError("Unsupported attn_mask dtype for Metal Flash Attention")
    if any(s < 0 for s in mask.stride()):
        mask = mask.contiguous()
    keep.append(mask)
    n = mask.dim()
    shape = (ctypes.c_int64 * n)(*mask.shape)
    strides = (ctypes.c_int64 * n)(*mask.stride())
    span = 1 + sum((d - 1) * s for d, s in zip(mask.shape, mask.stride()) if d > 0)
    keep += [shape, strides]
    return [ctypes.c_void_p(mask.data_ptr()), span * mask.element_size(), shape, strides, n, mtype, scalar]


def _forward(query, key, value, mask, is_causal, scale, want_lse, out_dtype, window=-1):
    """Enqueue the dense forward on torch's current stream.  Returns (O [out_dtype], L fp32 or None)."""
    ctx = _context(query.device)
    B, H, Sq, D = query.shape
    Skv = key.size(2)
    q, k, v = (t if t.is_contiguous() else t.contiguous() for t in (query, key, value))
    out = torch.empty((B, H, Sq, D), device=query.device, dtype=out_dtype)
    lse = torch.empty((B, H, Sq), device=query.device, dtype=torch.float32) if want_lse else None
    keep = []
    margs = _mask_args(mask, query, keep)
    stream = ctypes.c_void_p(torch.cuda.current_stream(query.device).cuda_stream or 0)
    with _Bound(ctx) as bind:
        rc = _lib.mfa_attention_forward_ex(ctx.handle, bind(q), bind(k), bind(v), bind(out), bind(lse),
                                           B, Sq, Skv, H, D, float(scale), bool(is_causal), int(window),
                                           _PREC[query.dtype], _PREC[out_dtype], *margs, _stream_arg(stream, query))
    if rc != 0:
        raise RuntimeError(f"Metal Flash Attention forward failed with code {rc}: {_ffi._get_error_string(rc)}")
    return out, lse


def _stream_arg(stream, t):
    """A NULL stream pointer would mean "block on the library stream": the legacy default stream is passed as
    cudaStreamLegacy (0x1) so the call stays an enqueue."""
    return stream if stream.value else ctypes.c_void_p(1)


def _backward(d_out, query, key, value, out_fp32, lse, mask, is_causal, scale, window=-1):
    ctx = _context(query.device)
    B, H, Sq, D = query.shape
    Skv = key.size(2)
    d_out = d_out.to(query.dtype).contiguous()
    dq = torch.empty(query.shape, device=query.device, dtype=torch.float32)
    dk = torch.empty(key.shape, device=query.device, dtype=torch.float32)
    dv = torch.empty(value.shape, device=query.device, dtype=torch.float32)
    dbuf = torch.empty((B * H * Sq,), device=query.device, dtype=torch.float32)
    keep = []
    margs = _mask_args(mask, query, keep)
    stream = ctypes.c_void_p(torch.cuda.current_stream(query.device).cuda_stream or 0)
    with _Bound(ctx) as bind:
        rc = _lib.mfa_attention_backward_ex(ctx.handle, bind(d_out), bind(query), bind(key), bind(value),
                                            bind(out_fp32), bind(lse), bind(dq), bind(dk), bind(dv), bind(dbuf),
                                            B, Sq, Skv, H, D, float(scale), bool(is_causal), int(window),
                                            _PREC[query.dtype], *margs, _stream_arg(stream, query))
    if rc != 0:
        raise RuntimeError(f"MetalFlashAttention backward failed with code {rc}")
    return dq, dk, dv


class MetalFlashAttentionFn(torch.autograd.Function):
    """metal_sdpa_backend.cpp:2672-2861: forward saves (q, k, v, O fp32, L); backward returns grads in q's dtype."""

    @staticmethod
    def forward(ctx, query, key, value, is_causal, scale, attn_mask=None):
        q, k, v = query.contiguous(), key.contiguous(), value.contiguous()
        out32, lse = _forward(q, k, v, attn_mask, is_causal, scale, True, torch.float32)
        ctx.save_for_backward(q, k, v, out32, lse)
        ctx.mask, ctx.is_causal, ctx.scale = attn_mask, bool(is_causal), float(scale)
        return out32 if query.dtype == torch.float32 else out32.to(query.dtype)

    @staticmethod
    def backward(ctx, d_output):
        q, k, v, out32, lse = ctx.saved_tensors
        dq, dk, dv = _backward(d_output, q, k, v, out32, lse, ctx.mask, ctx.is_causal, ctx.scale)
        if q.dtype != torch.float32:
            dq, dk, dv = dq.to(q.dtype), dk.to(q.dtype), dv.to(q.dtype)
        return dq, dk, dv, None, None, None


def metal_flash_attention_autograd(query, key, value, is_causal=False, scale=0.0, attn_mask=None):
    """scale <= 0 means 1/sqrt(head_dim), as in the reference binding's default (python_bindings.cpp:77-84)."""
    _check_inputs(query, key, value)
    if not scale or scale <= 0.0:
        scale = 1.0 / math.sqrt(query.size(-1))
    return MetalFlashAttentionFn.apply(query, key, value, is_causal, scale, attn_mask)


def _thd_handle(bind, t):
    """[total, heads, D] tensor (unit stride along D) -> a [1, heads, total, D] strided handle over the same memory."""
    T, Hn, D = t.shape
    shape = (ctypes.c_int64 * 4)(1, Hn, T, D)
    strides = (ctypes.c_int64 * 4)(T * t.stride(0), t.stride(1), t.stride(0), t.stride(2))
    h = _ffi.mfa_buffer_t()
    nbytes = max(((T - 1) * t.stride(0) + (Hn - 1) * t.stride(1) + D) * t.element_size(), 1)
    _ffi._check_error(_lib.mfa_buffer_from_mtl_buffer_with_strides(bind.ctx.handle, ctypes.c_void_p(t.data_ptr()), nbytes,
                                                                   shape, strides, 4, ctypes.byref(h)))
    bind.handles.append(h)
    return h


class MetalFlashAttentionVarlenFn(torch.autograd.Function):
    """Packed variable-length attention: forward saves (q, k, v, O fp32 [Hq, total_q, D], L); dK / dV come back per KV head."""

    @staticmethod
    def forward(ctx, query, key, value, cu_q, cu_k, is_causal, scale, window):
        dev = query.device
        T, H, D = query.shape
        Tk, Hkv = key.shape[0], key.shape[1]
        out32 = torch.empty((H, T, D), device=dev, dtype=torch.float32)
        lse = torch.empty((H, T), device=dev, dtype=torch.float32)
        lib_ctx = _context(dev)
        stream = _stream_arg(ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream or 0), query)
        with _Bound(lib_ctx) as bind:
            rc = _lib.mfa_attention_forward_varlen(
                lib_ctx.handle, _thd_handle(bind, query), _thd_handle(bind, key), _thd_handle(bind, value), bind(out32),
                bind(lse), bind(cu_q), bind(cu_k), cu_q.numel() - 1, T, Tk, H, Hkv, D, float(scale), bool(is_causal),
                int(window), _PREC[query.dtype], _ffi.MFA_PRECISION_FP32, stream)
        if rc != 0:
            raise RuntimeError(f"Metal Flash Attention varlen forward failed with code {rc}: {_ffi._get_error_string(rc)}")
        ctx.save_for_backward(query, key, value, out32, lse, cu_q, cu_k)
        ctx.is_causal, ctx.scale, ctx.window = bool(is_causal), float(scale), int(window)
        out = out32.transpose(0, 1)
        return out.contiguous() if query.dtype == torch.float32 else out.to(query.dtype)

    @staticmethod
    def backward(ctx, d_output):
        query, key, value, out32, lse, cu_q, cu_k = ctx.saved_tensors
        dev = query.device
        T, H, D = query.shape
        Tk, Hkv = key.shape[0], key.shape[1]
        d_out = d_output.to(query.dtype).transpose(0, 1).contiguous()          # [H, total_q, D]
        dq = torch.empty((H, T, D), device=dev, dtype=torch.float32)
        dk = torch.empty((Hkv, Tk, D), device=dev, dtype=torch.float32)
        dv = torch.empty((Hkv, Tk, D), device=dev, dtype=torch.float32)
        dbuf = torch.empty((H * T,), device=dev, dtype=torch.float32)
        lib_ctx = _context(dev)
        stream = _stream_arg(ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream or 0), query)
        with _Bound(lib_ctx) as bind:
            rc = _lib.mfa_attention_backward_varlen(
                lib_ctx.handle, bind(d_out), _thd_handle(bind, query), _thd_handle(bind, key), _thd_handle(bind, value),
                bind(out32), bind(lse), bind(dq), bind(dk), bind(dv), bind(dbuf), bind(cu_q), bind(cu_k), cu_q.numel() - 1,
                T, Tk, H, Hkv, D, ctx.scale, ctx.is_causal, ctx.window, _PREC[query.dtype], stream)
        if rc != 0:
            raise RuntimeError(f"Metal Flash Attention varlen backward failed with code {rc}: {_ffi._get_error_string(rc)}")
        dq, dk, dv = (g.transpose(0, 1).to(query.dtype).contiguous() for g in (dq, dk, dv))
        return dq, dk, dv, None, None, None, None, None


def metal_flash_attention_varlen(q, k, v, cu_seqlens_q, cu_seqlens_k, is_causal=False, scale=None, window=-1):
    """Attention over sequences packed along the token axis, without a dense mask.  q is [total_q, Hq, D], k / v
    [total_k, Hkv, D] (Hkv divides Hq: grouped-query attention without copies of K / V); cu_seqlens_q / cu_seqlens_k are int32
    CUDA tensors of num_seqs + 1 offsets (0, non-decreasing, ending at total_q / total_k).  Query row i of segment s sees the keys
    of segment s only; is_causal and window (>= 0: keys more than `window` positions behind are hidden) apply to the positions
    inside the segment, top-left aligned.  Returns O [total_q, Hq, D] in q's dtype; differentiable in q, k, v.  Enqueued on
    torch's current stream.  A row that sees no key gets O = 0."""
    for t in (q, k, v):
        if not t.is_cuda or t.dim() != 3 or t.stride(-1) != 1:
            raise RuntimeError("metal_flash_attention_varlen: q, k, v must be 3-D CUDA tensors [total, heads, head_dim] "
                               "with unit stride along head_dim")
    if q.dtype not in _PREC or k.dtype != q.dtype or v.dtype != q.dtype:
        raise RuntimeError("metal_flash_attention_varlen: q, k, v must share one of float16, bfloat16, float32")
    if k.shape != v.shape or k.size(2) != q.size(2) or q.size(1) % k.size(1):
        raise RuntimeError(f"metal_flash_attention_varlen: shapes q={tuple(q.shape)} k={tuple(k.shape)} v={tuple(v.shape)}")
    for c in (cu_seqlens_q, cu_seqlens_k):
        if c.dtype != torch.int32 or c.dim() != 1 or c.device != q.device or not c.is_contiguous():
            raise RuntimeError("metal_flash_attention_varlen: cu_seqlens must be contiguous 1-D int32 tensors on q's device")
    if cu_seqlens_q.numel() != cu_seqlens_k.numel() or cu_seqlens_q.numel() < 2:
        raise RuntimeError("metal_flash_attention_varlen: cu_seqlens_q / cu_seqlens_k need the same num_seqs + 1 >= 2 entries")
    if scale is None or scale <= 0.0:
        scale = 1.0 / math.sqrt(q.size(-1))
    return MetalFlashAttentionVarlenFn.apply(q, k, v, cu_seqlens_q, cu_seqlens_k, is_causal, scale,
                                             -1 if window is None or window < 0 else int(window))


def _bshd_handle(bind, t):
    """[B, S, heads, D] tensor (unit stride along D) -> a [B, heads, S, D] strided handle over the same memory."""
    B, S, Hn, D = t.shape
    shape = (ctypes.c_int64 * 4)(B, Hn, S, D)
    strides = (ctypes.c_int64 * 4)(t.stride(0), t.stride(2), t.stride(1), t.stride(3))
    h = _ffi.mfa_buffer_t()
    nbytes = max(((B - 1) * t.stride(0) + (S - 1) * t.stride(1) + (Hn - 1) * t.stride(2) + D) * t.element_size(), 1)
    _ffi._check_error(_lib.mfa_buffer_from_mtl_buffer_with_strides(bind.ctx.handle, ctypes.c_void_p(t.data_ptr()), nbytes,
                                                                   shape, strides, 4, ctypes.byref(h)))
    bind.handles.append(h)
    return h


def _check_append_args(fn, q, k_cache, k, v, rotary_cos, rotary_sin):
    """Arguments of the cache append of the K/V-cache calls: k / v shaped like q with the caches' KV heads, fp32 rotary tables
    [rotary_rows, rotary_dim / 2] with rotary_dim a multiple of 16 up to D, and no tables without k / v."""
    if (k is None) != (v is None):
        raise RuntimeError(f"{fn}: k and v go together")
    if (rotary_cos is None) != (rotary_sin is None):
        raise RuntimeError(f"{fn}: rotary_cos and rotary_sin go together")
    if k is None:
        if rotary_cos is not None:
            raise RuntimeError(f"{fn}: rotary_cos / rotary_sin need k and v: the new tokens' keys are rotated on their way into "
                               "the cache, and q with them")
        return
    if torch.is_grad_enabled() and (k.requires_grad or v.requires_grad):
        raise RuntimeError(f"{fn} has no backward: call it under torch.no_grad() or on tensors that do not require grad")
    want = (*q.shape[:-2], k_cache.size(2) if k_cache.dim() == 4 else -1, q.size(-1))
    for name, t in (("k", k), ("v", v)):
        if tuple(t.shape) != want or t.dtype != q.dtype or t.device != q.device or t.stride(-1) != 1:
            raise RuntimeError(f"{fn}: {name} must be {want} in q's dtype on q's device with unit stride along head_dim, got "
                               f"{tuple(t.shape)} {t.dtype} on {t.device}")
    if rotary_cos is None:
        return
    if rotary_cos.dtype != torch.float32 or rotary_sin.dtype != torch.float32:
        raise RuntimeError(f"{fn}: rotary_cos / rotary_sin must be float32")
    if rotary_cos.dim() != 2 or rotary_cos.shape != rotary_sin.shape or rotary_cos.size(0) == 0:
        raise RuntimeError(f"{fn}: rotary_cos / rotary_sin must be [rotary_rows, rotary_dim / 2], got "
                           f"{tuple(rotary_cos.shape)} and {tuple(rotary_sin.shape)}")
    rd = 2 * rotary_cos.size(1)
    if rd == 0 or rd % 16 or rd > q.size(-1):
        raise RuntimeError(f"{fn}: rotary_dim = {rd} must be a multiple of 16 and at most head_dim = {q.size(-1)}")
    for t in (rotary_cos, rotary_sin):
        if t.device != q.device or not t.is_contiguous():
            raise RuntimeError(f"{fn}: rotary_cos / rotary_sin must be contiguous tensors on q's device")


def _append(bind, handle, stream, q, k, v, kch, vch, cu_seqlens_q, cache_seqlens, block_table, rotary_cos, rotary_sin,
            interleaved, B, T, max_sq, H, Hkv, D, cap, page, npages):
    """Enqueues mfa_kvcache_append; returns the Q the attention reads (rotated into a new tensor when there are tables)."""
    q_out = None if rotary_cos is None else torch.empty(q.shape, device=q.device, dtype=q.dtype)
    rows, rd = (0, 0) if rotary_cos is None else (rotary_cos.size(0), 2 * rotary_cos.size(1))
    rc = _lib.mfa_kvcache_append(
        bind.ctx.handle, None if q_out is None else handle(bind, q), None if q_out is None else handle(bind, q_out),
        handle(bind, k), handle(bind, v), kch, vch, bind(cu_seqlens_q), bind(cache_seqlens), bind(block_table), bind(rotary_cos),
        bind(rotary_sin), rows, rd, bool(interleaved), B, T, max_sq, H, Hkv, D, cap, page, npages, _PREC[q.dtype], stream)
    if rc != 0:
        raise RuntimeError(f"Metal Flash Attention kvcache append failed with code {rc}: {_ffi._get_error_string(rc)}")
    return q if q_out is None else q_out


def metal_flash_attention_with_kvcache(q, k_cache, v_cache, cache_seqlens, block_table=None, is_causal=True, scale=None,
                                       window=-1, return_lse=False, *, k=None, v=None, rotary_cos=None, rotary_sin=None,
                                       rotary_interleaved=False):
    """Attention of the Sq new tokens of each sequence against that sequence's K/V cache (inference decode, speculative
    decode, chunked prefill).  q is [B, Sq, H, D] (bf16 / fp16, D a multiple of 8 up to 128); k_cache / v_cache are
    [B, capacity, Hkv, D], or with block_table (int32 [B, capacity / page_size] page ids) paged pools
    [num_pages, page_size, Hkv, D] with page_size a multiple of 16.  Hkv divides H (grouped-query attention without copies).
    cache_seqlens (int32 [B]) counts the valid keys of each sequence, the new tokens included (write their K / V into the cache
    first); token s sits at position cache_seqlens[b] - Sq + s and is_causal / window are bottom-right aligned.  Returns O
    [B, Sq, H, D] in q's dtype (and L fp32 [B, H, Sq] in log2 units with return_lse).  Cache rows past cache_seqlens[b] inside
    the last 128-key tile (in a paged cache: rows of the pages that block_table points to there) are read and enter P V with
    weight 0, so they must hold finite values: allocate pools with torch.zeros, not torch.empty.  Enqueued on torch's current
    stream with no copies of q or the caches, so it can be captured in a CUDA graph after one call of the shape outside the
    capture; the graph stays valid when later calls of other shapes run.  Forward only.

    With k / v ([B, Sq, Hkv, D], the new tokens' keys and values) the call first writes them into the caches, in place, at rows
    cache_seqlens[b] - Sq + s, then runs the attention; both are enqueued on the current stream.  Unlike flash-attn's
    flash_attn_with_kvcache, cache_seqlens keeps its meaning here: the lengths after the append, the new tokens included.  With
    rotary_cos / rotary_sin (fp32 [rotary_rows, rotary_dim / 2], one angle per pair, rotary_dim a multiple of 16 up to D) K is
    rotated on its way into the cache and Q with it, both at their cache positions (table row = cache row): rotary_interleaved
    pairs (2i, 2i+1), otherwise the half-split pairs (i, i + rotary_dim / 2) of Llama / NeoX.  The rotated Q goes to a new tensor;
    q itself is not modified.  Rotary tables without k / v raise, as in flash-attn."""
    _check_append_args("metal_flash_attention_with_kvcache", q, k_cache, k, v, rotary_cos, rotary_sin)
    if torch.is_grad_enabled() and any(t.requires_grad for t in (q, k_cache, v_cache)):
        raise RuntimeError("metal_flash_attention_with_kvcache has no backward: call it under torch.no_grad() or on "
                           "tensors that do not require grad")
    for t in (q, k_cache, v_cache):
        if not t.is_cuda or t.dim() != 4 or t.stride(-1) != 1:
            raise RuntimeError("metal_flash_attention_with_kvcache: q, k_cache, v_cache must be 4-D CUDA tensors with unit "
                               "stride along head_dim")
    if q.dtype not in (torch.float16, torch.bfloat16) or k_cache.dtype != q.dtype or v_cache.dtype != q.dtype:
        raise RuntimeError("metal_flash_attention_with_kvcache: q, k_cache, v_cache must share float16 or bfloat16")
    B, Sq, H, D = q.shape
    if k_cache.shape != v_cache.shape or k_cache.size(3) != D or H % k_cache.size(2):
        raise RuntimeError(f"metal_flash_attention_with_kvcache: shapes q={tuple(q.shape)} k_cache={tuple(k_cache.shape)} "
                           f"v_cache={tuple(v_cache.shape)}")
    Hkv = k_cache.size(2)
    for name, t in (("cache_seqlens", cache_seqlens), ("block_table", block_table)):
        if t is not None and (t.dtype != torch.int32 or t.device != q.device or not t.is_contiguous()):
            raise RuntimeError(f"metal_flash_attention_with_kvcache: {name} must be a contiguous int32 tensor on q's device")
    if cache_seqlens.shape != (B,):
        raise RuntimeError(f"metal_flash_attention_with_kvcache: cache_seqlens must be [{B}], got {tuple(cache_seqlens.shape)}")
    if block_table is None:
        if k_cache.size(0) != B:
            raise RuntimeError(f"metal_flash_attention_with_kvcache: contiguous caches need batch {B}")
        cap, page, npages = k_cache.size(1), 0, 0
    else:
        if block_table.dim() != 2 or block_table.size(0) != B:
            raise RuntimeError("metal_flash_attention_with_kvcache: block_table must be [batch, pages per sequence]")
        if not (k_cache.is_contiguous() and v_cache.is_contiguous()):
            raise RuntimeError("metal_flash_attention_with_kvcache: paged pools must be contiguous")
        npages, page = k_cache.size(0), k_cache.size(1)
        cap = block_table.size(1) * page
    if scale is None or scale <= 0.0:
        scale = 1.0 / math.sqrt(D)
    out = torch.empty(q.shape, device=q.device, dtype=q.dtype)
    lse = torch.empty((B, H, Sq), device=q.device, dtype=torch.float32) if return_lse else None
    lib_ctx = _context(q.device)
    stream = _stream_arg(ctypes.c_void_p(torch.cuda.current_stream(q.device).cuda_stream or 0), q)
    with _Bound(lib_ctx) as bind:
        paged = block_table is not None
        kch = bind(k_cache) if paged else _bshd_handle(bind, k_cache)
        vch = bind(v_cache) if paged else _bshd_handle(bind, v_cache)
        if k is not None:
            q = _append(bind, _bshd_handle, stream, q, k, v, kch, vch, None, cache_seqlens, block_table, rotary_cos, rotary_sin,
                        rotary_interleaved, B, 0, Sq, H, Hkv, D, cap, page, npages)
        rc = _lib.mfa_attention_forward_kvcache(
            lib_ctx.handle, _bshd_handle(bind, q), kch, vch, _bshd_handle(bind, out), bind(lse), bind(cache_seqlens),
            bind(block_table), B, Sq, H, Hkv, D, cap, page, npages, float(scale), bool(is_causal),
            -1 if window is None or window < 0 else int(window), _PREC[q.dtype], _PREC[q.dtype], stream)
    if rc != 0:
        raise RuntimeError(f"Metal Flash Attention kvcache forward failed with code {rc}: {_ffi._get_error_string(rc)}")
    return (out, lse) if return_lse else out


def metal_flash_attention_varlen_with_kvcache(q, k_cache, v_cache, cu_seqlens_q, cache_seqlens, max_seqlen_q, block_table=None,
                                              is_causal=True, scale=None, window_size=None, return_lse=False, *, k=None, v=None,
                                              rotary_cos=None, rotary_sin=None, rotary_interleaved=False):
    """metal_flash_attention_with_kvcache with a per-sequence number of new tokens: one call for a continuous-batching step
    that mixes decodes, speculative runs and prefill chunks.  q is [total_q, H, D]; sequence b owns query rows
    cu_seqlens_q[b]:cu_seqlens_q[b+1] (int32 CUDA tensor of num_seqs + 1 offsets: 0, non-decreasing, ending at total_q), and
    row s of it sits at position cache_seqlens[b] - sq_b + s (is_causal / window_size bottom-right aligned).  Caches,
    block_table and cache_seqlens are those of metal_flash_attention_with_kvcache with batch = num_seqs.  max_seqlen_q is a Python
    int bounding every segment: it sizes the work, so nothing is read back from the device.  Returns O [total_q, H, D] in q's
    dtype (and L fp32 [H, total_q] in log2 units with return_lse).  Enqueued on torch's current stream with no copies of q or
    the caches; it can be captured in a CUDA graph after one call of the shape outside the capture, and replays may carry new
    cu_seqlens_q contents, cache lengths and cache contents.  Forward only.

    k / v ([total_q, Hkv, D]), rotary_cos / rotary_sin and rotary_interleaved append the new tokens' K / V (rotated) to the caches
    first, as in metal_flash_attention_with_kvcache: token s of sequence b goes to cache row and table row
    cache_seqlens[b] - sq_b + s, and cache_seqlens counts the new tokens (unlike flash-attn)."""
    _check_append_args("metal_flash_attention_varlen_with_kvcache", q, k_cache, k, v, rotary_cos, rotary_sin)
    if torch.is_grad_enabled() and any(t.requires_grad for t in (q, k_cache, v_cache)):
        raise RuntimeError("metal_flash_attention_varlen_with_kvcache has no backward: call it under torch.no_grad() or on "
                           "tensors that do not require grad")
    if isinstance(max_seqlen_q, bool) or not isinstance(max_seqlen_q, int) or max_seqlen_q < 1:
        raise RuntimeError("metal_flash_attention_varlen_with_kvcache: max_seqlen_q must be a Python int >= 1")
    if not q.is_cuda or q.dim() != 3 or q.stride(-1) != 1:
        raise RuntimeError("metal_flash_attention_varlen_with_kvcache: q must be a 3-D CUDA tensor [total_q, heads, head_dim] with "
                           "unit stride along head_dim")
    for t in (k_cache, v_cache):
        if not t.is_cuda or t.dim() != 4 or t.stride(-1) != 1:
            raise RuntimeError("metal_flash_attention_varlen_with_kvcache: k_cache, v_cache must be 4-D CUDA tensors with unit "
                               "stride along head_dim")
    if q.dtype not in (torch.float16, torch.bfloat16) or k_cache.dtype != q.dtype or v_cache.dtype != q.dtype:
        raise RuntimeError("metal_flash_attention_varlen_with_kvcache: q, k_cache, v_cache must share float16 or bfloat16")
    T, H, D = q.shape
    if k_cache.shape != v_cache.shape or k_cache.size(3) != D or H % k_cache.size(2):
        raise RuntimeError(f"metal_flash_attention_varlen_with_kvcache: shapes q={tuple(q.shape)} "
                           f"k_cache={tuple(k_cache.shape)} v_cache={tuple(v_cache.shape)}")
    Hkv = k_cache.size(2)
    for name, t in (("cu_seqlens_q", cu_seqlens_q), ("cache_seqlens", cache_seqlens), ("block_table", block_table)):
        if t is not None and (t.dtype != torch.int32 or t.device != q.device or not t.is_contiguous()):
            raise RuntimeError(f"metal_flash_attention_varlen_with_kvcache: {name} must be a contiguous int32 tensor on q's device")
    if cu_seqlens_q.dim() != 1 or cu_seqlens_q.numel() < 2:
        raise RuntimeError("metal_flash_attention_varlen_with_kvcache: cu_seqlens_q must hold num_seqs + 1 >= 2 offsets")
    B = cu_seqlens_q.numel() - 1
    if cache_seqlens.shape != (B,):
        raise RuntimeError(f"metal_flash_attention_varlen_with_kvcache: cache_seqlens must be [{B}], "
                           f"got {tuple(cache_seqlens.shape)}")
    if block_table is None:
        if k_cache.size(0) != B:
            raise RuntimeError(f"metal_flash_attention_varlen_with_kvcache: contiguous caches need batch {B}")
        cap, page, npages = k_cache.size(1), 0, 0
    else:
        if block_table.dim() != 2 or block_table.size(0) != B:
            raise RuntimeError("metal_flash_attention_varlen_with_kvcache: block_table must be [num_seqs, pages per sequence]")
        if not (k_cache.is_contiguous() and v_cache.is_contiguous()):
            raise RuntimeError("metal_flash_attention_varlen_with_kvcache: paged pools must be contiguous")
        npages, page = k_cache.size(0), k_cache.size(1)
        cap = block_table.size(1) * page
    if scale is None or scale <= 0.0:
        scale = 1.0 / math.sqrt(D)
    out = torch.empty(q.shape, device=q.device, dtype=q.dtype)
    lse = torch.empty((H, T), device=q.device, dtype=torch.float32) if return_lse else None
    lib_ctx = _context(q.device)
    stream = _stream_arg(ctypes.c_void_p(torch.cuda.current_stream(q.device).cuda_stream or 0), q)
    with _Bound(lib_ctx) as bind:
        paged = block_table is not None
        kch = bind(k_cache) if paged else _bshd_handle(bind, k_cache)
        vch = bind(v_cache) if paged else _bshd_handle(bind, v_cache)
        if k is not None:
            q = _append(bind, _thd_handle, stream, q, k, v, kch, vch, cu_seqlens_q, cache_seqlens, block_table, rotary_cos,
                        rotary_sin, rotary_interleaved, B, T, max_seqlen_q, H, Hkv, D, cap, page, npages)
        rc = _lib.mfa_attention_forward_kvcache_varlen(
            lib_ctx.handle, _thd_handle(bind, q), kch, vch, _thd_handle(bind, out), bind(lse), bind(cu_seqlens_q),
            bind(cache_seqlens), bind(block_table), B, T, max_seqlen_q, H, Hkv, D, cap, page, npages, float(scale),
            bool(is_causal), -1 if window_size is None or window_size < 0 else int(window_size), _PREC[q.dtype], _PREC[q.dtype],
            stream)
    if rc != 0:
        raise RuntimeError(f"Metal Flash Attention kvcache varlen forward failed with code {rc}: {_ffi._get_error_string(rc)}")
    return (out, lse) if return_lse else out


def _dense_mask_f32(mask, query, Skv):
    """The quantised entry points take NULL or a dense fp32 additive [B,H,Sq,Skv] mask (metal_sdpa_backend.cpp:3210-3231)."""
    if mask is None:
        return None
    B, H, Sq, _ = query.shape
    if mask.dtype == torch.bool:
        m = torch.zeros(mask.shape, device=query.device, dtype=torch.float32).masked_fill_(~mask.to(query.device), float("-inf"))
    else:
        m = mask.to(device=query.device, dtype=torch.float32)
    while m.dim() < 4:
        m = m.unsqueeze(0)
    return m.expand(B, H, Sq, Skv).contiguous()


class MetalQuantizedFlashAttentionFn(torch.autograd.Function):
    """metal_sdpa_backend.cpp:3139-3383: quantise on the device, attention on the integer codes, fp32 O / L / grads."""

    @staticmethod
    def forward(ctx, query, key, value, is_causal, scale, target_precision, quant_mode, attn_mask=None):
        mctx = _context(query.device)
        B, H, Sq, D = query.shape
        Skv = key.size(2)
        q, k, v = query.contiguous(), key.contiguous(), value.contiguous()
        mask = _dense_mask_f32(attn_mask, query, Skv)
        out = torch.empty((B, H, Sq, D), device=query.device, dtype=torch.float32)
        lse = torch.empty((B, H, Sq), device=query.device, dtype=torch.float32)
        torch.cuda.current_stream(query.device).synchronize()      # blocking entry point on the library's stream
        with _Bound(mctx) as bind:
            rc = _lib.mfa_quantized_forward_with_lse(mctx.handle, bind(q), bind(k), bind(v), bind(out), bind(lse),
                                                     bind(mask), B, Sq, Skv, H, D, float(scale), bool(is_causal),
                                                     int(target_precision), int(quant_mode), _PREC[query.dtype])
        if rc != 0:
            raise RuntimeError(f"Quantized Metal Flash Attention forward failed with code {rc}")
        ctx.save_for_backward(q, k, v, out, lse)
        ctx.mask = mask
        ctx.args = (bool(is_causal), float(scale), int(target_precision), int(quant_mode))
        return out if query.dtype == torch.float32 else out.to(query.dtype)

    @staticmethod
    def backward(ctx, d_output):
        q, k, v, out, lse = ctx.saved_tensors
        is_causal, scale, tp, mode = ctx.args
        mctx = _context(q.device)
        B, H, Sq, D = q.shape
        Skv = k.size(2)
        g = d_output.to(torch.float32).contiguous()               # grad_out is fp32 (MFABridge+Quantized.swift:365)
        dq = torch.empty(q.shape, device=q.device, dtype=torch.float32)
        dk = torch.empty(k.shape, device=q.device, dtype=torch.float32)
        dv = torch.empty(v.shape, device=q.device, dtype=torch.float32)
        torch.cuda.current_stream(q.device).synchronize()
        with _Bound(mctx) as bind:
            rc = _lib.mfa_quantized_backward(mctx.handle, bind(q), bind(k), bind(v), bind(out), bind(g), bind(lse),
                                             bind(dq), bind(dk), bind(dv), bind(ctx.mask), B, Sq, Skv, H, D, scale,
                                             is_causal, tp, mode, _PREC[q.dtype])
        if rc != 0:
            raise RuntimeError(f"Quantized Metal Flash Attention backward failed with code {rc}")
        if q.dtype != torch.float32:
            dq, dk, dv = dq.to(q.dtype), dk.to(q.dtype), dv.to(q.dtype)
        return dq, dk, dv, None, None, None, None, None


def metal_quantized_flash_attention_autograd(query, key, value, is_causal=False, scale=0.0, target_precision=QUANT_INT8,
                                             quant_mode=QUANT_TENSOR_WISE, attn_mask=None):
    _check_inputs(query, key, value)
    if target_precision not in (QUANT_INT8, QUANT_INT4):
        raise RuntimeError("target_precision must be 3 (INT8) or 4 (INT4)")
    if quant_mode not in (QUANT_TENSOR_WISE, QUANT_BLOCK_WISE):
        raise RuntimeError("quant_mode must be 0 (tensor-wise) or 2 (block-wise)")
    if not scale or scale <= 0.0:
        scale = 1.0 / math.sqrt(query.size(-1))
    return MetalQuantizedFlashAttentionFn.apply(query, key, value, is_causal, scale, target_precision, quant_mode,
                                                attn_mask)


def set_quantization_mode(precision: int, block_mode: int) -> None:
    """Route every F.scaled_dot_product_attention call through the INT8/INT4 path (python_bindings.cpp:98-102)."""
    if precision not in (QUANT_INT8, QUANT_INT4):
        raise RuntimeError("precision must be QUANT_INT8 or QUANT_INT4")
    if block_mode not in (QUANT_TENSOR_WISE, QUANT_BLOCK_WISE):
        raise RuntimeError("block_mode must be QUANT_TENSOR_WISE or QUANT_BLOCK_WISE")
    _quant["precision"], _quant["block_mode"] = int(precision), int(block_mode)


def clear_quantization_mode() -> None:
    _quant["precision"], _quant["block_mode"] = QUANT_NONE, QUANT_TENSOR_WISE


def get_dispatch_stats() -> dict:
    return dict(_stats)


def reset_dispatch_stats() -> None:
    for k in _STAT_KEYS:
        _stats[k] = 0


def metal_scaled_dot_product_attention(query, key, value, attn_mask=None, dropout_p=0.0, is_causal=False, scale=None,
                                       enable_gqa=False):
    """The SDPA entry (metal_sdpa_backend.cpp:1643-1904): 2-D / 3-D inputs are promoted to 4-D BHSD, GQA expands K/V,
    all-true bool masks are dropped, quantisation mode and requires_grad pick the autograd Functions; everything else
    is one asynchronous forward in the input dtype."""
    if key.dim() != value.dim() or key.dim() < 2 or key.size(-2) != value.size(-2):
        raise RuntimeError("Metal SDPA: key and value must have matching sequence lengths")
    if 2 <= query.dim() < 4 and key.dim() == query.dim():
        extra = 4 - query.dim()
        q4, k4, v4 = query, key, value
        for _ in range(extra):
            q4, k4, v4 = q4.unsqueeze(0), k4.unsqueeze(0), v4.unsqueeze(0)
        out = metal_scaled_dot_product_attention(q4, k4, v4, attn_mask, dropout_p, is_causal, scale, enable_gqa)
        for _ in range(extra):
            out = out.squeeze(0)
        return out
    _stats["total"] += 1
    _check_inputs(query, key, value)
    if dropout_p and dropout_p > 0.0:
        raise RuntimeError("Dropout not supported in Metal Flash Attention")
    key, value = _expand_gqa(query, key, value)
    sm_scale = float(scale) if scale is not None else 1.0 / math.sqrt(query.size(-1))
    mask = attn_mask
    if mask is not None and mask.dtype == torch.bool and mask.numel() > 0 and bool(mask.all()):
        _stats["mask_all_true_skipped"] += 1
        mask = None
    if _quant["precision"] != QUANT_NONE:
        _stats["quantized_autograd"] += 1
        return metal_quantized_flash_attention_autograd(query, key, value, is_causal, sm_scale, _quant["precision"],
                                                        _quant["block_mode"], mask)
    if torch.is_grad_enabled() and (query.requires_grad or key.requires_grad or value.requires_grad):
        _stats["fp32_autograd"] += 1
        return MetalFlashAttentionFn.apply(query, key, value, is_causal, sm_scale, mask)
    _stats["direct"] += 1
    out, _ = _forward(query, key, value, mask, is_causal, sm_scale, False, query.dtype)
    return out


def quantized_scaled_dot_product_attention(query, key, value, precision="int8", is_causal=False, scale=None):
    """python_bindings.cpp:132-141: runtime-quantised forward, per-tensor scales."""
    tp = {"int8": QUANT_INT8, "int4": QUANT_INT4}.get(str(precision).lower())
    if tp is None:
        raise RuntimeError(f"Unsupported quantization precision: {precision}")
    _check_inputs(query, key, value)
    sm_scale = float(scale) if scale is not None else 1.0 / math.sqrt(query.size(-1))
    with torch.no_grad():
        return MetalQuantizedFlashAttentionFn.apply(query, key, value, is_causal, sm_scale, tp, QUANT_TENSOR_WISE, None)


def hadamard_rotate(tensor: torch.Tensor, block_size: int) -> torch.Tensor:
    """In-place group-wise Hadamard rotation of an fp32 CUDA tensor (metal_sdpa_backend.cpp:3395-3420)."""
    if tensor.dtype != torch.float32 or not tensor.is_cuda or not tensor.is_contiguous():
        raise RuntimeError("hadamard_rotate expects a contiguous float32 CUDA tensor")
    if block_size <= 0 or tensor.numel() % block_size:
        raise RuntimeError("Tensor size not divisible by block_size")
    ctx = _context(tensor.device)
    torch.cuda.current_stream(tensor.device).synchronize()
    with _Bound(ctx) as bind:
        rc = _lib.mfa_hadamard_rotate(bind(tensor), int(block_size), tensor.numel() // int(block_size))
    if rc != 0:
        raise RuntimeError("Hadamard rotation failed")
    return tensor


def _rope_tables(table, B, S, D, device):
    """pair-duplicated fp32 [S,D] / [1,S,D] / [B,S,D] -> (contiguous fp32 [b,S,D], table_batch_stride): the table contract of
    mfa_rope_rotate_encode_mtl (MFABridge.swift:282,305: element b * stride + s * D + 2 * pair, stride 0 or S * D)."""
    t = table.to(device=device, dtype=torch.float32)
    if t.dim() == 2:
        t = t.unsqueeze(0)
    if t.dim() != 3 or t.size(1) != S or t.size(2) != D or t.size(0) not in (1, B):
        raise RuntimeError("rope tables must be [S,D], [1,S,D] or [B,S,D]")
    return t.contiguous(), (S * D if t.size(0) == B and B > 1 else 0)


def _rope(x, cos_t, sin_t, negate_sin=False):
    ctx = _context(x.device)
    B, H, S, D = x.shape
    cos_f, bstride = _rope_tables(cos_t, B, S, D, x.device)
    sin_f, _ = _rope_tables(sin_t, B, S, D, x.device)
    dst = torch.empty((B, H, S, D), device=x.device, dtype=x.dtype)
    prec = {torch.float16: b"fp16", torch.bfloat16: b"bf16", torch.float32: b"fp32"}[x.dtype]
    stream = ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream or 0)
    if x.stride(3) != 1:
        x = x.contiguous()
    rc = _lib.mfa_rope_rotate_encode_mtl(ctx.handle, _stream_arg(stream, x), ctypes.c_void_p(x.data_ptr()), 0,
                                         x.stride(0), x.stride(1), x.stride(2), ctypes.c_void_p(dst.data_ptr()), 0,
                                         ctypes.c_void_p(cos_f.data_ptr()), 0, ctypes.c_void_p(sin_f.data_ptr()), 0,
                                         bstride, bool(negate_sin), B, H, S, D, prec)
    if rc != 0:
        raise RuntimeError(f"RoPE rotation failed with code {rc}")
    return dst


class RopeRotateFn(torch.autograd.Function):
    """Interleaved-pair rotary embedding with its exact backward: the rotation is orthonormal, so the gradient of the input
    is the inverse rotation (negate_sin) of the gradient of the output -- the reference adapter's dQ / dK transform
    (metal_sdpa_backend.cpp:2883-3122, MFABridge.swift:262-267)."""

    @staticmethod
    def forward(ctx, x, cos_t, sin_t):
        ctx.save_for_backward(cos_t, sin_t)
        return _rope(x, cos_t, sin_t)

    @staticmethod
    def backward(ctx, grad):
        cos_t, sin_t = ctx.saved_tensors
        return _rope(grad.contiguous(), cos_t, sin_t, negate_sin=True), None, None


def rope_scaled_dot_product_attention(query, key, value, rope_cos, rope_sin, attn_mask=None, is_causal=False, scale=None):
    """Interleaved-pair RoPE of Q and K on the device, then the SDPA entry (metal_sdpa_backend.cpp:1440-1560); gradients
    flow back through the attention backward and the inverse rotation of dQ / dK."""
    _check_inputs(query, key, value)
    if query.size(2) != key.size(2):
        raise RuntimeError("rope_scaled_dot_product_attention expects equal query / key sequence lengths")
    q_r, k_r = RopeRotateFn.apply(query, rope_cos, rope_sin), RopeRotateFn.apply(key, rope_cos, rope_sin)
    return metal_scaled_dot_product_attention(q_r, k_r, value, attn_mask, 0.0, is_causal, scale)


def is_metal_available() -> bool:
    return bool(_lib.mfa_is_device_supported())


def has_native_bfloat() -> bool:
    return _lib.mfa_has_native_bfloat() != 0


def has_native_bfloat_msl32() -> bool:
    return _lib.mfa_has_native_bfloat_msl32() != 0


def get_version():
    a, b, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    _lib.mfa_get_version(ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
    return (a.value, b.value, c.value)
