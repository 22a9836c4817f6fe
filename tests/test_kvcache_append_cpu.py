"""CPU tests of the K/V-cache append (mfa_kvcache_append): NULL handles, bad geometry and bad rotary arguments are argument
errors, a valid call without a device reports MFA_ERROR_DEVICE_NOT_SUPPORTED (never a crash, never a CPU fallback), the torch
adapters reject malformed append arguments, and the kernel keeps everything in registers."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

INVALID_ARGS, DEVICE_NOT_SUPPORTED = 1, 3
BF16, FP32 = 1, 2
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _call(lib, ctx, bufs, *, q=True, cu=True, table=True, rot=True, rows=64, rd=64, n=2, T=5, msq=4, H=8, Hkv=2, D=64,
          cap=256, page=16, pages=32, prec=BF16):
    """bufs: [k_new, v_new, k_cache, v_cache, cache_seqlens] handles; h stands in for every optional one that is set."""
    h = bufs[0]
    return lib.mfa_kvcache_append(ctx, h if q else None, h if q else None, *bufs[:4], h if cu else None, bufs[4],
                                  h if table else None, h if rot else None, h if rot else None, rows, rd, False, n, T, msq, H,
                                  Hkv, D, cap, page, pages, prec, None)


def _placeholder():
    keep = np.zeros(4096, np.uint8)
    return keep, ctypes.c_void_p(keep.ctypes.data)


def test_append_null_handles_are_invalid_args():
    from umfa import _ffi
    lib = _ffi._lib
    keep, h = _placeholder()
    assert _call(lib, None, [h] * 5) == INVALID_ARGS
    for i in range(5):                              # k_new, v_new, k_cache, v_cache, cache_seqlens
        bufs = [h] * 5
        bufs[i] = None
        assert _call(lib, h, bufs) == INVALID_ARGS, i
    assert _call(lib, h, [h] * 5, table=False) == INVALID_ARGS                  # paged without a block table
    assert _call(lib, h, [h] * 5, page=0, pages=0) == INVALID_ARGS              # contiguous with a block table
    assert lib.mfa_kvcache_append(h, h, None, h, h, h, h, h, h, h, h, h, 64, 64, False, 2, 5, 4, 8, 2, 64, 256, 16, 32,
                                  BF16, None) == INVALID_ARGS                   # q without q_out
    assert lib.mfa_kvcache_append(h, h, h, h, h, h, h, h, h, h, h, None, 64, 64, False, 2, 5, 4, 8, 2, 64, 256, 16, 32,
                                  BF16, None) == INVALID_ARGS                   # cos without sin


@pytest.mark.parametrize("kw", [
    dict(rot=False, rd=0),          # rotating q needs tables
    dict(rot=False, q=False, rd=16),                 # rotary_dim without tables
    dict(rd=0),                     # tables without rotary_dim
    dict(rd=24),                    # rotary_dim not a multiple of 16
    dict(rd=80),                    # rotary_dim above head_dim
    dict(rows=0),                   # empty tables
    dict(page=24),                  # page_size not a multiple of 16
    dict(cap=264),                  # capacity not a multiple of the page
    dict(H=8, Hkv=3),
    dict(prec=FP32),                # caches are bf16 / fp16
    dict(D=136, rd=64),             # head_dim above 128
    dict(D=60, rd=48),              # head_dim not a multiple of 8
    dict(n=0),
    dict(T=0),
    dict(msq=0),
    dict(msq=6),                    # max_seqlen_q above total_q
    dict(cu=False, n=65535, msq=40000),              # more tokens than one launch takes
])
def test_append_bad_arguments_are_invalid_args(kw):
    from umfa import _ffi
    lib = _ffi._lib
    keep, h = _placeholder()
    kw.setdefault("table", kw.get("page", 16) != 0)
    assert _call(lib, h, [h] * 5, **kw) == INVALID_ARGS


def test_append_without_device_reports_it():
    import umfa
    from umfa import _ffi
    if umfa.is_metal_available():
        pytest.skip("a GPU is present")
    lib = _ffi._lib
    keep, h = _placeholder()
    assert _call(lib, h, [h] * 5) == DEVICE_NOT_SUPPORTED
    assert _call(lib, h, [h] * 5, q=False) == DEVICE_NOT_SUPPORTED                                # K only
    assert _call(lib, h, [h] * 5, q=False, rot=False, rd=0, rows=0) == DEVICE_NOT_SUPPORTED       # no rotation
    assert _call(lib, h, [h] * 5, cu=False, table=False, page=0, pages=0) == DEVICE_NOT_SUPPORTED


def test_umfa_append_argument_validation():
    from umfa import core
    ctx = None                                      # every check runs before the context is used
    kn = np.zeros((2, 3, 2, 64), np.uint16)
    kc = np.zeros((2, 64, 2, 64), np.uint16)
    cos = np.zeros((64, 32), np.float32)
    with pytest.raises(ValueError, match="go together"):
        core.kvcache_append(ctx, kn, kn, kc, kc, [5, 6], rotary_cos=cos)
    with pytest.raises(ValueError, match="float32"):
        core.kvcache_append(ctx, kn, kn, kc, kc, [5, 6], rotary_cos=cos.astype(np.float64), rotary_sin=cos.astype(np.float64))
    with pytest.raises(ValueError, match="multiple of 16"):
        core.kvcache_append(ctx, kn, kn, kc, kc, [5, 6], rotary_cos=cos[:, :12], rotary_sin=cos[:, :12])
    with pytest.raises(ValueError, match="needs rotary"):
        core.kvcache_append(ctx, kn, kn, kc, kc, [5, 6], q=np.zeros((2, 3, 8, 64), np.uint16))
    with pytest.raises(ValueError, match="C-contiguous"):
        core.kvcache_append(ctx, kn, kn, kc[:, ::2], kc[:, ::2], [5, 6])
    with pytest.raises(ValueError, match="k_new / v_new must be"):
        core.kvcache_append(ctx, kn, kn[:, :2], kc, kc, [5, 6])


def test_torch_adapters_reject_malformed_append_arguments():
    torch = pytest.importorskip("torch")
    from pytorch_custom_op_ffi import metal_flash_attention_varlen_with_kvcache as fv
    from pytorch_custom_op_ffi import metal_flash_attention_with_kvcache as f
    q = torch.zeros(2, 3, 8, 64, dtype=torch.bfloat16)
    kc = torch.zeros(2, 128, 2, 64, dtype=torch.bfloat16)
    k = torch.zeros(2, 3, 2, 64, dtype=torch.bfloat16)
    lens = torch.tensor([4, 9], dtype=torch.int32)
    cos = torch.zeros(128, 32)
    with pytest.raises(RuntimeError, match="need k and v"):
        f(q, kc, kc, lens, rotary_cos=cos, rotary_sin=cos)
    with pytest.raises(RuntimeError, match="go together"):
        f(q, kc, kc, lens, k=k)
    with pytest.raises(RuntimeError, match="go together"):
        f(q, kc, kc, lens, k=k, v=k, rotary_cos=cos)
    with pytest.raises(RuntimeError, match="float32"):
        f(q, kc, kc, lens, k=k, v=k, rotary_cos=cos.double(), rotary_sin=cos.double())
    with pytest.raises(RuntimeError, match=r"\[rotary_rows"):
        f(q, kc, kc, lens, k=k, v=k, rotary_cos=cos, rotary_sin=cos[:64])
    with pytest.raises(RuntimeError, match="multiple of 16"):
        f(q, kc, kc, lens, k=k, v=k, rotary_cos=cos[:, :4], rotary_sin=cos[:, :4])
    with pytest.raises(RuntimeError, match="multiple of 16"):
        f(q, kc, kc, lens, k=k, v=k, rotary_cos=torch.zeros(128, 40), rotary_sin=torch.zeros(128, 40))
    with pytest.raises(RuntimeError, match="k must be"):
        f(q, kc, kc, lens, k=k[:, :2], v=k, rotary_cos=cos, rotary_sin=cos)
    with pytest.raises(RuntimeError, match="v must be"):
        f(q, kc, kc, lens, k=k, v=k.half())
    qv = torch.zeros(5, 8, 64, dtype=torch.bfloat16)
    cu = torch.tensor([0, 1, 5], dtype=torch.int32)
    with pytest.raises(RuntimeError, match="need k and v"):
        fv(qv, kc, kc, cu, lens, 4, rotary_cos=cos, rotary_sin=cos)
    with pytest.raises(RuntimeError, match="k must be"):
        fv(qv, kc, kc, cu, lens, 4, k=k, v=k)
    # valid append arguments reach the adapter's own checks (CPU tensors are rejected there)
    with pytest.raises(RuntimeError, match="CUDA"):
        fv(qv, kc, kc, cu, lens, 4, k=torch.zeros(5, 2, 64, dtype=torch.bfloat16), v=torch.zeros(5, 2, 64, dtype=torch.bfloat16),
           rotary_cos=cos, rotary_sin=cos)


def test_append_kernel_has_no_stack_frame():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    obj = os.path.join(ROOT, "universal-metal-flash-attention_b200", "lib", "kvcache_append.o")
    if not os.path.exists(cuobjdump) or not os.path.exists(obj):
        pytest.skip("cuobjdump or the object files are not available")
    out = subprocess.run([cuobjdump, "-res-usage", obj], capture_output=True, text=True).stdout
    seen = set()
    for m in re.finditer(r"Function \S*kvcache_append_kernelI(\S+?)EEv\S*:\s*\n\s*REG:(\d+) STACK:(\d+)", out):
        assert int(m.group(3)) == 0, m.group(0)
        seen.add(m.group(1))
    assert seen == {"6__half", "13__nv_bfloat16"}, seen
