"""CPU tests of the boundary: the library loads, exports every symbol the headers declare, prototypes match the
reference header, and the no-device error behaviour follows the reference bridge."""
import ctypes
import json
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INCLUDE = os.path.join(ROOT, "include")
# prototypes and probe output of the reference's Sources/MFAFFI/include/mfa_ffi.h (tests/golden/make_reference_abi.py)
REF_ABI = os.path.join(ROOT, "tests", "golden", "reference_abi.json")
PROBE = r'''
#include <stdio.h>
#include <stddef.h>
#include HDR
int main(void){
  printf("%d %d %d %d %d %d\n", MFA_SUCCESS, MFA_ERROR_INVALID_ARGS, MFA_ERROR_MEMORY_ALLOCATION,
         MFA_ERROR_DEVICE_NOT_SUPPORTED, MFA_ERROR_KERNEL_COMPILATION, MFA_ERROR_EXECUTION_FAILED);
  printf("%d %d %d %d %d\n", MFA_PRECISION_FP16, MFA_PRECISION_BF16, MFA_PRECISION_FP32, MFA_PRECISION_INT8, MFA_PRECISION_INT4);
  printf("%d %d %d | %d %d %d %d\n", MFA_MASK_TYPE_NONE, MFA_MASK_TYPE_BOOL, MFA_MASK_TYPE_ADDITIVE,
         MFA_MASK_SCALAR_BYTE, MFA_MASK_SCALAR_FP16, MFA_MASK_SCALAR_BF16, MFA_MASK_SCALAR_FP32);
  printf("%d %d %d\n", MFA_QUANT_KERNEL_FORWARD, MFA_QUANT_KERNEL_BACKWARD_QUERY, MFA_QUANT_KERNEL_BACKWARD_KEY_VALUE);
  printf("%zu %zu %zu %zu %zu\n", sizeof(mfa_quantized_layout_t), offsetof(mfa_quantized_layout_t, qScale),
         offsetof(mfa_quantized_layout_t, maskBuffer), offsetof(mfa_quantized_layout_t, scratch1),
         offsetof(mfa_quantized_layout_t, qBlockScales));
  printf("%zu %zu %zu\n", sizeof(mfa_quantized_capabilities_t), offsetof(mfa_quantized_capabilities_t, max_heads),
         offsetof(mfa_quantized_capabilities_t, max_block_size));
  printf("%zu %zu %zu %zu\n", sizeof(mfa_error_t), sizeof(mfa_precision_t), sizeof(mfa_context_t), sizeof(mfa_mla_context_t));
  return 0; }
'''


def _lib():
    from umfa import _ffi
    return _ffi


def _strip_comments(text):
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    return re.sub(r"//[^\n]*", " ", text)


def _prototypes(text):
    """name -> normalised 'ret(argtype,argtype,...)' for every mfa_* function declaration."""
    text = _strip_comments(text)
    out = {}
    for m in re.finditer(r"([A-Za-z_][\w\s\*]*?)\b(mfa_\w+)\s*\(([^;{}]*?)\)\s*;", text, flags=re.S):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        norm = []
        for a in args.split(","):
            a = " ".join(a.split())
            if a in ("void", ""):
                continue
            a = re.sub(r"\b([A-Za-z_]\w*)$", "", a).strip() if not a.endswith("*") and " " in a else a
            norm.append(a.replace(" *", "*").replace("* ", "*"))
        out[name] = (" ".join(ret.split()).replace("extern ", ""), tuple(norm))
    return out


def test_library_exports_every_declared_symbol():
    ffi = _lib()
    declared = set()
    for h in ("mfa_ffi.h", "mfa_ffi_ext.h"):
        declared |= set(_prototypes(open(os.path.join(INCLUDE, h)).read()))
    assert len(declared) >= 29 + 13
    lib = ctypes.CDLL(ffi.library_path())
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, missing
    assert set(ffi.SIGNATURES) == declared


def test_exports_only_mfa_symbols():
    from umfa import _ffi
    out = subprocess.run(["nm", "-D", "--defined-only", _ffi.library_path()], capture_output=True, text=True).stdout
    names = [l.split()[-1] for l in out.splitlines() if l.strip()]
    assert names and all(n.startswith("mfa_") for n in names)


def probe_output(header, tmp_dir):
    """What PROBE prints when compiled against `header`: enum values, struct sizes and offsets."""
    src = os.path.join(tmp_dir, "probe.c")
    exe = os.path.join(tmp_dir, "probe")
    with open(src, "w") as f:
        f.write(PROBE)
    subprocess.run(["/usr/bin/gcc", "-std=c11", f'-DHDR="{os.path.abspath(header)}"', src, "-o", exe], check=True)
    return subprocess.run([exe], capture_output=True, text=True, check=True).stdout


def _reference_abi():
    with open(REF_ABI) as f:
        return json.load(f)


def test_header_matches_reference_prototypes():
    ours = _prototypes(open(os.path.join(INCLUDE, "mfa_ffi.h")).read())
    ref = {name: (ret, tuple(args)) for name, (ret, args) in _reference_abi()["prototypes"].items()}
    assert set(ref) == set(ours)
    for name, proto in ref.items():
        assert ours[name] == proto, name


def test_header_enums_and_structs_match_reference(tmp_path):
    """Compile the probe against our header and compare what it prints with the reference header's output."""
    assert probe_output(os.path.join(INCLUDE, "mfa_ffi.h"), str(tmp_path)) == _reference_abi()["probe"]


def test_headers_compile_as_c_and_cxx(tmp_path):
    src = tmp_path / "t.c"
    src.write_text('#include "mfa_ffi_ext.h"\nint main(void){ return (int)sizeof(mfa_quantized_layout_t) == 0; }\n')
    subprocess.run(["/usr/bin/gcc", "-std=c99", "-Wall", "-Werror", "-I", INCLUDE, "-c", str(src), "-o", str(tmp_path / "t.o")], check=True)
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", "-Werror", "-x", "c++", "-I", INCLUDE, "-c", str(src), "-o", str(tmp_path / "t2.o")], check=True)


def test_error_strings_and_version():
    ffi = _lib()
    # MFABridge.swift:1528-1536 / Tests/MFAFFITests/MFAFFITests.swift:42-51
    expect = {0: "Success", 1: "Invalid arguments", 2: "Memory allocation failed", 3: "Device not supported",
              4: "Kernel compilation failed", 5: "Execution failed", 99: "Unknown error", -1: "Unknown error"}
    for code, text in expect.items():
        assert ffi._get_error_string(code) == text
    import umfa
    assert umfa.get_version() == (1, 0, 0)


def test_null_arguments_return_invalid_args():
    ffi = _lib()
    L = ffi._lib
    assert L.mfa_create_context(None) == 1
    assert L.mfa_create_buffer(None, 16, None) == 1
    assert L.mfa_buffer_contents(None) is None
    L.mfa_destroy_buffer(None)
    L.mfa_destroy_context(None)
    assert L.mfa_get_gpu_latency(None) == 0.0
    z = [0] * 5
    rc = L.mfa_attention_forward(None, None, None, None, None, *z, 1.0, False, 0, 0, 0, False, False, False, False,
                                 None, 0, None, None, 0, 0, 0)
    assert rc == 1            # NULL handle -> MFA_ERROR_INVALID_ARGS (MFABridge.swift:1105-1110)
    assert L.mfa_attention_backward(None, *[None] * 10, *z, 1.0, False, 0, 0, False, False, False, False) == 1
    assert L.mfa_hadamard_rotate(None, 8, 1) == 1


def test_layout_and_capabilities_constants():
    ffi = _lib()
    buf = (ctypes.c_int32 * 38)(*([7] * 38))
    ffi._lib.mfa_get_quantized_layout(0, buf)
    assert list(buf) == [-1] * 38          # QuantizedLayoutManifest+FFI.swift:146-155
    cap = (ctypes.c_uint8 * 16)()
    ffi._lib.mfa_get_quantized_capabilities(cap)
    assert cap[0] == 1 and cap[1] == 1


def test_stubs_outside_hot_path():
    ffi = _lib()
    h = ctypes.c_void_p()
    assert ffi._lib.mfa_mla_create_context(ctypes.byref(h)) == 0 and h.value
    assert ffi._lib.mfa_mla_init_weights(h, 1, 1, 1) == 3
    ffi._lib.mfa_mla_destroy_context(h)
    assert ffi._lib.mfa_sparse_indexer_scores(None, None, None, 1, 1, 1, 1, 8, 1.0, None, None) == 3


def test_no_device_means_error_not_fallback():
    """Without an sm_100 GPU the product path must fail loudly (code 3), never compute on the CPU."""
    import umfa
    if umfa.is_metal_available():
        pytest.skip("a GPU is present")
    with pytest.raises(umfa.MFAError) as e:
        umfa.MFAContext()
    assert e.value.code == 3


def test_python_adapter_argument_validation():
    import umfa
    from umfa import core
    with pytest.raises(ValueError):
        core._parse_precision("fp64")
    with pytest.raises(TypeError):
        core._dims([1], [2], [3], "bshd")
    q = np.zeros((4, 8), np.float32)
    with pytest.raises(ValueError):
        core._dims(q, np.zeros((4, 9), np.float32), np.zeros((4, 8), np.float32), "bshd")
    d = core._dims(np.zeros((2, 5, 3, 8)), np.zeros((2, 7, 3, 8)), np.zeros((2, 7, 3, 8)), "bshd")
    assert (d.B, d.H, d.Sq, d.Skv, d.D, d.bshd) == (2, 3, 5, 7, 8, True)
    m = core._prepare_mask_metadata(np.ones((5, 7), bool), (2, 3, 5, 7))
    assert m.mask_type == 1 and m.ndim == 2 and list(m.shape) == [5, 7] and list(m.strides) == [7, 1]
    with pytest.raises(ValueError):
        core._prepare_mask_metadata(np.ones((4, 7), bool), (2, 3, 5, 7))


def test_c_program_links_by_library_name_and_runs(tmp_path):
    """A plain C consumer, the way the reference's Rust / ObjC examples link (-lMFAFFI, examples/rust-ffi/build.rs:45;
    extern calls as in examples/objc/simple_bridge.m:23-35): version, error string ownership (free), and a context request
    that either succeeds (GPU present) or reports MFA_ERROR_DEVICE_NOT_SUPPORTED -- never a crash, never a CPU fallback."""
    lib_dir = os.path.join(ROOT, "universal-metal-flash-attention_b200", "lib")
    src = tmp_path / "consumer.c"
    src.write_text(r'''
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "mfa_ffi.h"
int main(void) {
  int major = -1, minor = -1, patch = -1;
  mfa_get_version(&major, &minor, &patch);
  if (major != 1 || minor != 0 || patch != 0) return 10;
  char* s = (char*)mfa_error_string(MFA_ERROR_INVALID_ARGS);
  if (!s || strcmp(s, "Invalid arguments") != 0) return 11;
  free(s);                                             /* strdup'd by the library: the caller frees */
  mfa_context_t ctx = NULL;
  mfa_error_t rc = mfa_create_context(&ctx);
  if (mfa_is_device_supported()) {
    if (rc != MFA_SUCCESS || !ctx) return 12;
    mfa_buffer_t b = NULL;
    if (mfa_create_buffer(ctx, 1024, &b) != MFA_SUCCESS || !mfa_buffer_contents(b)) return 13;
    mfa_destroy_buffer(b);
    mfa_destroy_context(ctx);
  } else if (rc != MFA_ERROR_DEVICE_NOT_SUPPORTED) {
    return 14;
  }
  if (mfa_attention_forward(NULL, NULL, NULL, NULL, NULL, 1, 1, 1, 1, 8, 1.0f, false, MFA_PRECISION_FP32, MFA_PRECISION_FP32,
                            MFA_PRECISION_FP32, false, false, false, false, NULL, 0, NULL, NULL, 0, MFA_MASK_TYPE_NONE,
                            MFA_MASK_SCALAR_BYTE) != MFA_ERROR_INVALID_ARGS) return 15;
  puts("c consumer ok");
  return 0;
}
''')
    exe = tmp_path / "consumer"
    subprocess.run(["/usr/bin/gcc", "-std=c99", "-Wall", "-Werror", "-I", INCLUDE, str(src), "-o", str(exe), "-L", lib_dir,
                    "-lMFAFFI", "-Wl,-rpath," + lib_dir], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "c consumer ok" in r.stdout, (r.returncode, r.stdout, r.stderr)


def test_headline_forward_instantiations_do_not_spill():
    """The unmasked bf16 / fp16 / fp32-split / int8 forward instantiations must keep O and S in registers: a stack frame in them
    cost 6 % of the headline number once (an epilogue branch indexed the O registers dynamically; round 2)."""
    import re
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    obj = os.path.join(ROOT, "universal-metal-flash-attention_b200", "lib", "attn_fwd_tc.o")
    if not os.path.exists(cuobjdump) or not os.path.exists(obj):
        pytest.skip("cuobjdump or the object file is not available")
    out = subprocess.run([cuobjdump, "-res-usage", obj], capture_output=True, text=True).stdout
    seen = set()
    for m in re.finditer(r"Function (\S*fwd_tc_kernelILi(\d+)ELi(\d+)ELi0E\S*):\s*\n\s*REG:(\d+) STACK:(\d+)", out):
        d, mode, stack = int(m.group(2)), int(m.group(3)), int(m.group(5))
        if mode in (0, 1, 3, 4, 8):          # f16, bf16, int8 + e4m3, fp32 split, wide bf16
            seen.add((d, mode))
            assert stack == 0, (m.group(1), stack)
    assert seen == {(64, 0), (128, 0), (64, 1), (128, 1), (128, 3), (128, 4), (128, 8)}, seen


def test_staged_mask_instantiations_exist_and_do_not_spill():
    """The instantiations that stage external-mask tiles in shared memory (MASKED = 2: forward bf16 / fp16 at both head-dim
    widths, both backward kernels) are in the library and keep their working set in registers."""
    import re
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    lib_dir = os.path.join(ROOT, "universal-metal-flash-attention_b200", "lib")
    if not os.path.exists(cuobjdump) or not os.path.exists(os.path.join(lib_dir, "attn_fwd_tc.o")):
        pytest.skip("cuobjdump or the object files are not available")
    fwd = subprocess.run([cuobjdump, "-res-usage", os.path.join(lib_dir, "attn_fwd_tc.o")], capture_output=True, text=True).stdout
    seen = set()
    for m in re.finditer(r"Function \S*fwd_tc_kernelILi(\d+)ELi([01])ELi2E\S*:\s*\n\s*REG:(\d+) STACK:(\d+)", fwd):
        assert int(m.group(4)) == 0, m.group(0)
        seen.add((int(m.group(1)), int(m.group(2))))
    assert seen == {(64, 0), (64, 1), (128, 0), (128, 1)}
    bwd = subprocess.run([cuobjdump, "-res-usage", os.path.join(lib_dir, "attn_bwd_tc.o")], capture_output=True, text=True).stdout
    seen = set()
    for m in re.finditer(r"Function \S*bwd_(dkv|dq)_tc_kernelILi(\d+)ELb([01])ELi2E\S*:\s*\n\s*REG:(\d+) STACK:(\d+)", bwd):
        assert int(m.group(5)) == 0, m.group(0)
        seen.add((m.group(1), int(m.group(2)), int(m.group(3))))
    assert len(seen) == 8, seen
