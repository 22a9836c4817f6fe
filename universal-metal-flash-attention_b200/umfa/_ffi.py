"""ctypes bindings to libMFAFFI.so (the B200 build of the MFAFFI C ABI).

Host-side mirror of the reference's examples/python-ffi/src/umfa/_ffi.py: same constants, MFAError and
_check_error; the only intended difference is the library file name (.so next to this package, or
$MFA_LIBRARY) -- the reference hard-codes libMFAFFI.dylib (_ffi.py:57-90 there).
There is no fallback: if the library is missing, importing this module raises.
"""
import ctypes
import os
from pathlib import Path

MFA_SUCCESS = 0
MFA_ERROR_INVALID_ARGS = 1
MFA_ERROR_MEMORY_ALLOCATION = 2
MFA_ERROR_DEVICE_NOT_SUPPORTED = 3
MFA_ERROR_KERNEL_COMPILATION = 4
MFA_ERROR_EXECUTION_FAILED = 5

MFA_PRECISION_FP16 = 0
MFA_PRECISION_BF16 = 1
MFA_PRECISION_FP32 = 2
MFA_PRECISION_INT8 = 3
MFA_PRECISION_INT4 = 4

MFA_MASK_TYPE_NONE = 0
MFA_MASK_TYPE_BOOL = 1
MFA_MASK_TYPE_ADDITIVE = 2

MFA_MASK_SCALAR_BYTE = 0
MFA_MASK_SCALAR_FP16 = 1
MFA_MASK_SCALAR_BF16 = 2
MFA_MASK_SCALAR_FP32 = 3

mfa_error_t = ctypes.c_int32
mfa_precision_t = ctypes.c_int32
mfa_context_t = ctypes.c_void_p
mfa_buffer_t = ctypes.c_void_p


class MFAError(Exception):
    def __init__(self, code: int, message: str = ""):
        self.code = code
        self.message = message or _get_error_string(code)
        super().__init__(f"MFA Error {code}: {self.message}")


def library_path() -> str:
    env = os.environ.get("MFA_LIBRARY")
    if env:
        return env
    here = Path(__file__).resolve().parent
    for cand in (here.parent / "lib" / "libMFAFFI.so", Path("/usr/local/lib/libMFAFFI.so")):
        if cand.exists():
            return str(cand)
    raise RuntimeError("libMFAFFI.so not found -- run `python universal-metal-flash-attention_b200/build.py`")


_c = ctypes
_ctx, _buf, _u32, _u16, _i32, _f32, _b, _sz, _vp, _i64, _u64 = (
    _c.c_void_p, _c.c_void_p, _c.c_uint32, _c.c_uint16, _c.c_int32, _c.c_float, _c.c_bool, _c.c_size_t, _c.c_void_p,
    _c.c_int64, _c.c_uint64)
_pi64 = _c.POINTER(_c.c_int64)
_DIMS = [_u32, _u32, _u32, _u32, _u16]                  # batch, seq_q, seq_kv, heads, head_dim
_MASK = [_vp, _sz, _pi64, _pi64, _u32, _i32, _i32]     # ptr, bytes, shape, strides, ndim, type, scalar
_VARLEN = [_u32, _u32, _u32, _u32, _u32, _u16]         # num_seqs, total_q, total_k, heads, kv heads, head_dim
_QPARAMS = [_f32, _i32, _f32, _i32, _f32, _i32]
_T4 = [_b, _b, _b, _b]

# name -> (restype, argtypes); spelled exactly as include/mfa_ffi.h / mfa_ffi_ext.h declare them
SIGNATURES = {
    "mfa_get_quantized_layout": (None, [_i32, _vp]),
    "mfa_get_quantized_capabilities": (None, [_vp]),
    "mfa_create_context": (_i32, [_c.POINTER(_ctx)]),
    "mfa_destroy_context": (None, [_ctx]),
    "mfa_create_buffer": (_i32, [_ctx, _sz, _c.POINTER(_buf)]),
    "mfa_buffer_from_ptr": (_i32, [_ctx, _vp, _sz, _c.POINTER(_buf)]),
    "mfa_buffer_from_ptr_with_strides": (_i32, [_ctx, _vp, _sz, _pi64, _pi64, _u32, _c.POINTER(_buf)]),
    "mfa_buffer_from_mtl_buffer": (_i32, [_ctx, _vp, _sz, _c.POINTER(_buf)]),
    "mfa_buffer_from_mtl_buffer_with_strides": (_i32, [_ctx, _vp, _sz, _pi64, _pi64, _u32, _c.POINTER(_buf)]),
    "mfa_buffer_contents": (_vp, [_buf]),
    "mfa_destroy_buffer": (None, [_buf]),
    "mfa_attention_forward": (_i32, [_ctx, _buf, _buf, _buf, _buf] + _DIMS + [_f32, _b, _i32, _i32, _i32] + _T4 + _MASK),
    "mfa_attention_forward_str": (_i32, [_ctx, _buf, _buf, _buf, _buf] + _DIMS + [_f32, _b, _c.c_char_p, _c.c_char_p,
                                                                                _c.c_char_p] + _T4 + _MASK),
    "mfa_attention_encode_mtl": (_i32, [_ctx, _vp, _vp, _i64, _pi64, _vp, _i64, _pi64, _vp, _i64, _pi64, _vp, _i64,
                                        _vp, _i64, _pi64, _pi64, _u32, _i32, _i32] + _DIMS + [_f32, _b, _c.c_char_p,
                                                                                              _c.c_char_p]),
    "mfa_attention_forward_quantized": (_i32, [_ctx, _buf, _buf, _buf, _buf] + _DIMS + [_f32, _b] + _QPARAMS +
                                        [_i32, _i32, _i32, _i32] + _T4),
    "mfa_attention_forward_quantized_unified": (_i32, [_ctx, _buf, _buf, _buf, _buf] + _DIMS + [_f32, _b] + _QPARAMS +
                                                [_i32, _i32, _i32, _i32, _i32, _u32, _u32, _u32, _b, _b] + _T4),
    "mfa_attention_forward_quantized_enhanced": (_i32, [_ctx, _buf, _buf, _buf, _buf] + _DIMS + [_f32, _b] + _QPARAMS +
                                                 [_i32, _i32, _i32, _i32, _i32, _u32, _u32, _u32, _b, _b] + _T4),
    "mfa_attention_forward_quantized_direct": (_i32, [_ctx, _buf, _buf, _buf, _buf] + _DIMS + [_f32, _b] + _QPARAMS +
                                               [_i32, _i32, _i32, _i32] + _T4),
    "mfa_multihead_attention_quantized_direct": (_i32, [_ctx, _buf, _buf, _buf, _buf] + _DIMS + [_f32, _b] + _QPARAMS +
                                                 [_i32, _i32, _i32]),
    "mfa_sparse_indexer_scores": (_i32, [_ctx, _buf, _buf, _u32, _u32, _u32, _u32, _u16, _f32, _buf, _c.POINTER(_buf)]),
    "mfa_attention_backward": (_i32, [_ctx] + [_buf] * 10 + _DIMS + [_f32, _b, _i32, _i32] + _T4),
    "mfa_error_string": (_vp, [_i32]),
    "mfa_is_device_supported": (_b, []),
    "mfa_get_version": (None, [_c.POINTER(_c.c_int)] * 3),
    "mfa_get_gpu_latency": (_c.c_double, [_ctx]),
    "mfa_attention_backward_query_quantized": (_i32, [_ctx] + [_buf] * 8 + _DIMS + _QPARAMS + [_i32, _i32, _i32, _b] + _T4),
    "mfa_attention_backward_kv_quantized": (_i32, [_ctx] + [_buf] * 8 + _DIMS + _QPARAMS + [_i32, _i32, _i32, _b] + _T4),
    "mfa_attention_backward_query_quantized_ex": (_i32, [_ctx] + [_buf] * 8 + [_u32, _u32, _u32, _u32, _u32, _u16] +
                                                  _QPARAMS + [_i32, _i32, _i32, _b] + _T4 + [_buf] * 6 +
                                                  [_u32, _u32, _u32, _u32]),
    "mfa_attention_backward_kv_quantized_ex": (_i32, [_ctx] + [_buf] * 8 + [_u32, _u32, _u32, _u32, _u32, _u16] +
                                               _QPARAMS + [_i32, _i32, _i32, _b] + _T4 + [_buf] * 6 +
                                               [_u32, _u32, _u32, _u32]),
    "mfa_mla_create_context": (_i32, [_c.POINTER(_vp)]),
    "mfa_mla_destroy_context": (None, [_vp]),
    "mfa_mla_init_weights": (_i32, [_vp, _u32, _u32, _u32]),
    "mfa_mla_load_weights": (_i32, [_vp, _buf, _buf]),
    "mfa_mla_forward": (_i32, [_vp, _ctx, _buf, _c.POINTER(_buf), _c.POINTER(_buf), _u32, _u32, _u32, _u32, _u32]),
    # exported-but-undeclared in the reference header (mfa_ffi_ext.h part 1)
    "mfa_set_scale_arrays": (_i32, [_ctx, _c.POINTER(_f32), _u32, _c.POINTER(_f32), _u32, _c.POINTER(_f32), _u32]),
    "mfa_has_native_bfloat": (_i32, []),
    "mfa_has_native_bfloat_msl32": (_i32, []),
    "mfa_attention_forward_with_lse": (_i32, [_ctx, _buf, _buf, _buf, _buf, _buf] + _DIMS + [_f32, _b, _i32, _i32] + _T4),
    "mfa_quantized_forward_with_lse": (_i32, [_ctx] + [_buf] * 6 + _DIMS + [_f32, _b, _i32, _i32, _i32]),
    "mfa_quantized_backward": (_i32, [_ctx] + [_buf] * 10 + _DIMS + [_f32, _b, _i32, _i32, _i32]),
    "mfa_hadamard_rotate": (_i32, [_buf, _u32, _u32]),
    "mfa_rope_rotate_encode_mtl": (_c.c_int, [_ctx, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _vp, _i64,
                                             _i64, _b, _u32, _u32, _u32, _u32, _c.c_char_p]),
    # additive B200 symbols (mfa_ffi_ext.h part 2)
    "mfa_attention_forward_ex": (_i32, [_ctx, _buf, _buf, _buf, _buf, _buf] + _DIMS + [_f32, _b, _i32, _i32, _i32] +
                                 _MASK + [_vp]),
    "mfa_attention_forward_accumulate": (_i32, [_ctx, _buf, _buf, _buf, _buf, _buf] + _DIMS + [_f32, _b, _i32, _i32, _u32, _u32, _vp]),
    "mfa_attention_backward_ex": (_i32, [_ctx] + [_buf] * 10 + _DIMS + [_f32, _b, _i32, _i32] + _MASK + [_vp]),
    "mfa_attention_forward_varlen": (_i32, [_ctx] + [_buf] * 7 + _VARLEN + [_f32, _b, _i32, _i32, _i32, _vp]),
    "mfa_attention_backward_varlen": (_i32, [_ctx] + [_buf] * 12 + _VARLEN + [_f32, _b, _i32, _i32, _vp]),
    "mfa_attention_forward_kvcache": (_i32, [_ctx] + [_buf] * 7 + [_u32, _u32, _u32, _u32, _u16, _u32, _u32, _u32] +
                                      [_f32, _b, _i32, _i32, _i32, _vp]),
    "mfa_attention_forward_kvcache_varlen": (_i32, [_ctx] + [_buf] * 8 + [_u32, _u32, _u32, _u32, _u32, _u16, _u32, _u32, _u32] +
                                             [_f32, _b, _i32, _i32, _i32, _vp]),
    "mfa_kvcache_append": (_i32, [_ctx] + [_buf] * 11 + [_u32, _u16, _b, _u32, _u32, _u32, _u32, _u32, _u16, _u32, _u32, _u32,
                                                        _i32, _vp]),
    "mfa_quantize": (_i32, [_ctx, _buf, _buf, _buf, _u64, _u64, _u32, _u32, _i32, _i32, _f32, _vp]),
    "mfa_dequantize": (_i32, [_ctx, _buf, _buf, _buf, _u64, _u64, _u32, _u32, _i32, _vp]),
    "mfa_merge_partials": (_i32, [_ctx, _buf, _buf, _buf, _buf, _u64, _u32, _vp]),
    "mfa_ring_transport_available": (_b, []),
    "mfa_ring_get_unique_id": (_i32, [_vp, _sz]),
    "mfa_ring_create": (_i32, [_ctx, _vp, _sz, _i32, _i32, _c.POINTER(_vp)]),
    "mfa_ring_create_from_comm": (_i32, [_ctx, _vp, _i32, _i32, _c.POINTER(_vp)]),
    "mfa_ring_destroy": (None, [_vp]),
    "mfa_ring_transport": (_i32, [_vp]),
    "mfa_ring_handle_bytes": (_sz, []),
    "mfa_ring_prepare": (_i32, [_vp, _u32, _u32, _u32, _u16]),
    "mfa_ring_export_handles": (_i32, [_vp, _vp, _sz]),
    "mfa_ring_import_handles": (_i32, [_vp, _vp, _sz]),
    "mfa_ring_launch_count": (_u64, [_vp]),
    "mfa_ring_attention_forward": (_i32, [_vp, _buf, _buf, _buf, _buf, _buf, _u32, _u32, _u32, _u16, _f32, _i32, _vp]),
    "mfa_ring_attention_backward": (_i32, [_vp] + [_buf] * 9 + [_u32, _u32, _u32, _u16, _f32, _i32, _vp]),
    "mfa_set_quantized_pv_precision": (_i32, [_ctx, _i32]),
    "mfa_get_quantized_pv_precision": (_i32, [_ctx]),
    "mfa_set_device": (_i32, [_i32]),
    "mfa_get_device_count": (_i32, []),
    "mfa_last_kernel_name": (_c.c_char_p, [_ctx]),
    "mfa_launch_count": (_u64, [_ctx]),
}


def _load_library():
    lib = ctypes.CDLL(library_path())
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = the library does not export the ABI
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = _load_library()
_libc = ctypes.CDLL(None)
_libc.free.argtypes = [ctypes.c_void_p]


def _get_error_string(code: int) -> str:
    p = _lib.mfa_error_string(code)
    if not p:
        return "Unknown error"
    try:
        return ctypes.string_at(p).decode()
    finally:
        _libc.free(p)          # strdup'd by the library: the caller frees (mfa_ffi.h)


def _check_error(code: int) -> None:
    if code != MFA_SUCCESS:
        raise MFAError(code)
