// tc_host.h -- host-side helpers shared by the tcgen05 kernels: TMA tensor-map construction for [B, H, S, D] operand
// views (cuTensorMapEncodeTiled resolved through the runtime so the library loads without libcuda at link time).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdlib>
#include <mutex>

#include "common.h"

namespace mfa {
namespace tc {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qr) == cudaSuccess &&
        qr == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
    else
      cudaGetLastError();
  });
  return fn;
}

// [B, Hn, S, D] view with unit inner stride -> 4-D tensor map, box = (128 bytes of a row) x box_rows rows, 128B
// swizzle.  elem_bytes: 2 for fp16/bf16, 1 for int8/fp8 operands (box is then 128 elements wide), 4 for the fp32 output
// map of the forward's TMA-store epilogue (box = 32 floats).
inline bool make_map(CUtensorMap* out, const TensorView& t, int dtype, int B, int Hn, int S, int D, int box_rows = 128) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  const cuuint64_t eb = (dtype == kI8) ? 1 : (dtype == kF32) ? 4 : 2;
  cuuint64_t dims[4] = {(cuuint64_t)D, (cuuint64_t)S, (cuuint64_t)Hn, (cuuint64_t)B};
  cuuint64_t st[3] = {(cuuint64_t)t.ss * eb, (cuuint64_t)t.sh * eb, (cuuint64_t)t.sb * eb};
  if (Hn == 1) st[1] = st[0] * (cuuint64_t)S;
  if (B == 1) st[2] = st[1] * (cuuint64_t)Hn;
  // the box is always 128 bytes wide (one swizzle span): a head dim that is not a multiple of it leaves part of the last box out of
  // bounds, which TMA zero-fills on loads and clips on stores
  cuuint32_t box[4] = {(cuuint32_t)(128 / eb), (cuuint32_t)box_rows, 1, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  const CUtensorMapDataType ty = dtype == kBF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                               : dtype == kF16  ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                               : dtype == kF32  ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                                : CU_TENSOR_MAP_DATA_TYPE_UINT8;
  CUresult r = fn(out, ty, 4, const_cast<void*>(t.ptr), dims, st, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// packed bytes [B, Hn, S, row_bytes] contiguous (int4 codes, two per byte) -> 4-D tensor map, box = row_bytes x 128 rows,
// NO swizzle: the tile lands row-major in shared memory, where a converter warp expands it (attn_fwd_tc.cu, int4 modes)
inline bool make_map_raw(CUtensorMap* out, const void* ptr, int B, int Hn, int S, int row_bytes) {
  EncodeTiledFn fn = encode_fn();
  if (!fn || row_bytes <= 0 || (row_bytes & 15)) return false;
  cuuint64_t dims[4] = {(cuuint64_t)row_bytes, (cuuint64_t)S, (cuuint64_t)Hn, (cuuint64_t)B};
  cuuint64_t st[3] = {(cuuint64_t)row_bytes, (cuuint64_t)row_bytes * S, (cuuint64_t)row_bytes * S * Hn};
  cuuint32_t box[4] = {(cuuint32_t)row_bytes, 128, 1, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void*>(ptr), dims, st, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// [slots][B][Hn][S][D] contiguous 16-bit operand -> 5-D tensor map (ring attention's visiting K/V pairs), same box / swizzle
typedef CUresult (*EncodeTiledFn5)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline bool make_map5(CUtensorMap* out, const void* base, int dtype, int slots, int B, int Hn, int S, int D) {
  EncodeTiledFn fn = encode_fn();
  if (!fn || slots < 1) return false;
  const cuuint64_t eb = 2;
  cuuint64_t dims[5] = {(cuuint64_t)D, (cuuint64_t)S, (cuuint64_t)Hn, (cuuint64_t)B, (cuuint64_t)slots};
  cuuint64_t st[4] = {(cuuint64_t)D * eb, (cuuint64_t)S * D * eb, (cuuint64_t)Hn * S * D * eb, (cuuint64_t)B * Hn * S * D * eb};
  cuuint32_t box[5] = {64, 128, 1, 1, 1};
  if (box[0] > (cuuint32_t)D) box[0] = (cuuint32_t)D;
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  const CUtensorMapDataType ty = dtype == kBF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = fn(out, ty, 5, const_cast<void*>(base), dims, st, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// Q of grouped-query attention, [B, H = Hkv * G, Sq, D] view with unit inner stride -> 5-D tensor map (D, Sq, G, Hkv, B), box
// (64, sqb, G, 1, 1), 128B swizzle: one box lands the sqb tokens of all G query heads of a KV head as rows g * sqb + s of a tile.
inline bool make_map_gqa(CUtensorMap* out, const TensorView& t, int dtype, int B, int Hkv, int G, int Sq, int D, int sqb) {
  EncodeTiledFn fn = encode_fn();
  if (!fn || sqb < 1 || G < 1 || sqb * G > 128) return false;
  const cuuint64_t eb = 2;
  cuuint64_t dims[5] = {(cuuint64_t)D, (cuuint64_t)Sq, (cuuint64_t)G, (cuuint64_t)Hkv, (cuuint64_t)B};
  cuuint64_t st[4] = {(cuuint64_t)t.ss * eb, (cuuint64_t)t.sh * eb, (cuuint64_t)t.sh * G * eb, (cuuint64_t)t.sb * eb};
  if (Sq == 1) st[0] = (cuuint64_t)D * eb;              // extent-1 dims: any valid stride (the view's may be 0)
  if (G == 1) st[1] = st[0] * (cuuint64_t)Sq;
  if (Hkv == 1) st[2] = st[1] * (cuuint64_t)G;
  if (B == 1) st[3] = st[2] * (cuuint64_t)Hkv;
  cuuint32_t box[5] = {64, (cuuint32_t)sqb, (cuuint32_t)G, 1, 1};
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  const CUtensorMapDataType ty = dtype == kBF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = fn(out, ty, 5, const_cast<void*>(t.ptr), dims, st, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// TMA needs a 16-byte aligned base, unit inner stride and 16-byte multiples for the outer strides.
inline bool view_ok(const TensorView& t, int64_t Hn, int64_t B, int elem_bytes = 2) {
  const int64_t q = 16 / elem_bytes;
  if (t.sd != 1) return false;
  if (reinterpret_cast<uintptr_t>(t.ptr) & 15) return false;
  if (t.ss <= 0 || (t.ss % q)) return false;
  if (Hn > 1 && (t.sh <= 0 || (t.sh % q))) return false;
  if (B > 1 && (t.sb <= 0 || (t.sb % q))) return false;
  return true;
}

// Dense external mask (unit key stride, one row of terms per query row) with 1-byte (bool) or 2-byte (fp16 / bf16 additive) elements
// -> 4-D tensor map over [MB, MH, Sq, Skv] (broadcast dims have extent 1), box = 128 bytes x 128 rows, 128-byte swizzle: the kernels
// stage 128 x 128 mask tiles in shared memory instead of reading them row by row.  False when the mask does not qualify (row
// broadcast, fp32 terms, rows that are not 16-byte multiples, MFA_DISABLE_MASK_TMA): the kernels then read it in place.
inline bool make_mask_map(CUtensorMap* out, const AttnParams& p) {
  if (p.mask_kind == kMaskNone || !p.mask || getenv("MFA_DISABLE_MASK_TMA") || p.mask_sq <= 0 || p.mask_sk != 1) return false;
  const bool one_byte = p.mask_kind == kMaskBool;
  if (!one_byte && p.mask_scalar != kMaskBF16 && p.mask_scalar != kMaskF16) return false;
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  const long long eb = one_byte ? 1 : 2, q = 16 / eb;
  if ((reinterpret_cast<uintptr_t>(p.mask) & 15) || (p.mask_sq % q) || (p.mask_sh % q) || (p.mask_sb % q) || p.mask_sh < 0 || p.mask_sb < 0)
    return false;
  const int MH = p.mask_sh ? p.H : 1, MB = p.mask_sb ? p.B : 1;
  cuuint64_t dims[4] = {(cuuint64_t)p.Skv, (cuuint64_t)p.Sq, (cuuint64_t)MH, (cuuint64_t)MB};
  cuuint64_t st[3] = {(cuuint64_t)(p.mask_sq * eb), (cuuint64_t)(p.mask_sh * eb), (cuuint64_t)(p.mask_sb * eb)};
  if (MH == 1) st[1] = st[0] * (cuuint64_t)p.Sq;
  if (MB == 1) st[2] = st[1] * (cuuint64_t)MH;
  cuuint32_t box[4] = {(cuuint32_t)(128 / eb), 128, 1, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  return fn(out, one_byte ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<void*>(p.mask), dims, st, box,
            es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace tc
}  // namespace mfa
