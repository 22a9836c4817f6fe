// quant.cu -- HBM-bound helper kernels: symmetric int8/int4 quantiser, dequantiser, LSE merge of attention
// partials, Hadamard rotation, RoPE, dtype conversion.
//
// Quantiser contract (bit-exact with oracle/attention_oracle.c, which restates
// metal-flash-attention/Sources/FlashAttention/GEMM/GEMMQuantization.swift:305-623 and
// GEMMRuntimeQuantization.swift:80-181):  scale = absmax / 127 (int8) or / 7 (int4) as an IEEE fp32 division,
// optionally floored; code = clamp(roundf(x / scale)) with an IEEE division and round-half-away-from-zero;
// int4 packs two codes per byte, flat element 2i in the low nibble, stored +8, odd tail padded with code 0.
// Where the reference needs two dispatches and a host round trip per tensor, the common granularities
// (per-row, per-token-block, per-head) are one fused kernel: absmax and quantise from the same cached tile,
// 16-byte vector loads, algorithmic traffic = read once + write codes.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math_constants.h>

#include <cstdlib>

#include "common.h"

namespace mfa {
namespace {

template <typename T> __device__ __forceinline__ float to_f32(T x);
template <> __device__ __forceinline__ float to_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ float to_f32<__half>(__half x) { return __half2float(x); }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 x) { return __bfloat162float(x); }

// 8 consecutive elements -> fp32 (16-byte loads for 2-byte types, 2 x 16 bytes for fp32)
template <typename T> struct Vec8 {
  static __device__ __forceinline__ void load(const T* p, float out[8]) {
    uint4 raw = *reinterpret_cast<const uint4*>(p);
    const T* e = reinterpret_cast<const T*>(&raw);
#pragma unroll
    for (int i = 0; i < 8; ++i) out[i] = to_f32<T>(e[i]);
  }
};
template <> struct Vec8<float> {
  static __device__ __forceinline__ void load(const float* p, float out[8]) {
    float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
    out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = a.w; out[4] = b.x; out[5] = b.y; out[6] = b.z; out[7] = b.w;
  }
};

__device__ __forceinline__ float make_scale(float amax, int bits, float floor_v) {
  float sc = __fdiv_rn(amax, bits == 8 ? 127.0f : 7.0f);
  if (floor_v > 0.f && !(sc > floor_v)) sc = floor_v;
  return sc;
}

// Same code as quant_code() without a division per element: t = x * (1 / scale) is within ~1.2e-5 of the correctly
// rounded quotient for |t| < 129 (and beyond that everything clamps alike), so round(t) equals round(x / scale) unless t sits
// within 1e-4 of a half-integer -- those rare elements take the exact division.  Bit-exact by construction.  (Measured: the
// apply pass of a 28 MB bf16 tensor 19.2 -> 17.2 us without the division, -> 14.0 us with the magic-number rounding and the
// byte-permute packing below (round 2); the read-only abs-max pass takes 7.6 us, so the rest of the gap is still the
// per-element convert / round / clamp / pack arithmetic, not memory.  A register-resident single-trip block variant was tried
// and was slower than the two-trip one: 24.4 vs 21 us.  A four-rows-per-warp D-term kernel first measured slower as well, 36.6 vs
// 24 us -- its 64-bit row / head divisions were the cost; with those moved into the grid shape it runs in 15.5 us, attn_simt.cu.)
__device__ __forceinline__ int quant_code_exact(float x, float scale, int bits) {
  const float lo = bits == 8 ? -128.f : -8.f, hi = bits == 8 ? 127.f : 7.f;
  return (int)fminf(fmaxf(roundf(__fdiv_rn(x, scale)), lo), hi);
}
// Eight codes at once.  The scale of a block is never below amax / 127 (amax / 7), so |t| <= 127 (7) up to rounding and the
// nearest integer needs no clamp: adding 1.5 * 2^23 rounds t to it in the mantissa (ties to even) -- one FADD instead of trunc /
// copysign / add / trunc, and the integer falls out of the bit pattern.  Elements within 1e-4 of a tie (where half-away-from-zero
// and the inexact product could disagree with the exact quotient), NaN / infinite t (d is NaN then) and any t outside the range
// the argument above promises take the exact rule; the eight tests are merged into ONE branch (a branch per element cost more
// than the arithmetic it guarded: ~16 instructions per element before this, profiles/r02bh_helpers_two.csv).
// (packed f32x2 arithmetic for the multiply and the three adds: IEEE round-to-nearest per lane, i.e. the same bits as the scalar
// instructions at half the issue slots -- the ncu capture of the block pass showed 66 % issue utilisation and 23 executed
// instructions per element, profiles/r02bp_ncu_quant_span.txt)
typedef unsigned long long qf32x2;
__device__ __forceinline__ qf32x2 qpack2(float lo, float hi) { qf32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void qunpack2(qf32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ qf32x2 qmul2(qf32x2 a, qf32x2 b) { qf32x2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ qf32x2 qadd2(qf32x2 a, qf32x2 b) { qf32x2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ qf32x2 qsub2(qf32x2 a, qf32x2 b) { qf32x2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }

__device__ __forceinline__ void quant_codes8(const float* x, float scale, float inv, int bits, int* q) {
  if (!(scale > 0.f)) {
#pragma unroll
    for (int i = 0; i < 8; ++i) q[i] = 0;
    return;
  }
  const qf32x2 inv2 = qpack2(inv, inv), mg = qpack2(12582912.f, 12582912.f);
  bool rare = false;
#pragma unroll
  for (int i = 0; i < 8; i += 2) {
    const qf32x2 t2 = qmul2(qpack2(x[i], x[i + 1]), inv2);
    const qf32x2 y2 = qadd2(t2, mg);
    const qf32x2 d2 = qsub2(t2, qsub2(y2, mg));                // distance to the nearest integer, in [-1/2, 1/2]
    float y0, y1, d0, d1;
    qunpack2(y2, y0, y1);
    qunpack2(d2, d0, d1);
    q[i] = __float_as_int(y0) - 0x4B400000;
    q[i + 1] = __float_as_int(y1) - 0x4B400000;
    // near a tie, or t not finite (d is NaN then).  |t| <= 127 (7) by construction of the scale, so no range test is needed for the
    // magic-number rounding itself
    rare |= !(fabsf(d0) <= 0.5f - 1e-4f) || !(fabsf(d1) <= 0.5f - 1e-4f);
  }
  if (rare) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float t = x[i] * inv;
      const float y = t + 12582912.f;
      const float d = t - (y - 12582912.f);
      if (!(fabsf(d) <= 0.5f - 1e-4f)) q[i] = quant_code_exact(x[i], scale, bits);
    }
  }
}
// low bytes of four ints -> one word (three byte permutes instead of four masks, three shifts and three ors)
__device__ __forceinline__ uint32_t pack4_bytes(int a, int b, int c, int d) {
  return __byte_perm(__byte_perm((uint32_t)a, (uint32_t)b, 0x0040), __byte_perm((uint32_t)c, (uint32_t)d, 0x0040), 0x5410);
}
__device__ __forceinline__ float inv_scale(float scale) { return scale > 0.f ? __frcp_rn(scale) : 0.f; }

__device__ __forceinline__ int quant_code(float x, float scale, int bits) {
  if (!(scale > 0.f)) return 0;
  float r = roundf(__fdiv_rn(x, scale));
  const float lo = bits == 8 ? -128.f : -8.f, hi = bits == 8 ? 127.f : 7.f;
  r = fminf(fmaxf(r, lo), hi);
  return (int)r;
}

// ---- fused path: each quantisation block is a contiguous span [e0, e1) of the flat tensor (block_cols == cols).
// One worker (warp if WARP else CTA) per block; pass 1 absmax, pass 2 re-reads the same lines from L1/L2.
// Requires: span start and length multiples of 8 and 16-byte aligned base (checked by the launcher).
template <typename T, int BITS, bool WARP>
__global__ void __launch_bounds__(256) quant_span_kernel(const T* __restrict__ src, uint8_t* __restrict__ codes,
                                                         float* __restrict__ scales, uint64_t rows, uint64_t cols,
                                                         uint32_t block_rows, uint64_t group_rows, uint32_t nb_per_group,
                                                         uint64_t nblocks, float floor_v) {
  __shared__ float red[8];
  const int nworker = WARP ? 32 : (int)blockDim.x;           // CTA variant: 256 threads (launcher)
  const int wid = WARP ? (threadIdx.x >> 5) : 0;
  const int lane = WARP ? (threadIdx.x & 31) : threadIdx.x;
  const uint64_t blk = WARP ? (uint64_t)blockIdx.x * 8 + wid : blockIdx.x;
  if (blk >= nblocks) return;
  // (the block index fits 32 bits whenever the grid does: 32-bit division; inside the block everything is a 32-bit offset from the
  // block's own base pointers -- the span is at most 65536 elements -- instead of 64-bit element indices into the tensor.  The ncu
  // capture of this pass showed it instruction-bound, profiles/r02bp_ncu_quant_span.txt; the int8 call as a whole did not move with
  // this change, 0.309 vs 0.308 ms, profiles/r02br_bench_quant.json, so the index arithmetic was not the larger part of it)
  uint64_t g, lb;
  if (blk <= 0xffffffffull) { const uint32_t b32 = (uint32_t)blk; g = b32 / nb_per_group; lb = b32 % nb_per_group; }
  else { g = blk / nb_per_group; lb = blk % nb_per_group; }
  const uint64_t r0 = g * group_rows + lb * block_rows;
  uint64_t r1 = r0 + block_rows;
  if (r1 > (g + 1) * group_rows) r1 = (g + 1) * group_rows;
  if (r1 > rows) r1 = rows;
  const uint64_t e0 = r0 * cols;
  const uint32_t n = (uint32_t)((r1 - r0) * cols), step = (uint32_t)nworker * 8;
  const T* bsrc = src + e0;
  uint8_t* bcodes = codes + (BITS == 8 ? e0 : (e0 >> 1));

  float amax = 0.f;
  for (uint32_t e = (uint32_t)lane * 8; e < n; e += step) {
    float x[8];
    Vec8<T>::load(bsrc + e, x);
#pragma unroll
    for (int i = 0; i < 8; ++i) amax = fmaxf(amax, fabsf(x[i]));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  if (!WARP) {
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = amax;
    __syncthreads();
    amax = red[0];
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) amax = fmaxf(amax, red[i]);
  }
  const float sc = make_scale(amax, BITS, floor_v);
  const float inv = inv_scale(sc);
  if (lane == 0) scales[blk] = sc;

  for (uint32_t e = (uint32_t)lane * 8; e < n; e += step) {
    float x[8];
    Vec8<T>::load(bsrc + e, x);
    int q[8];
    quant_codes8(x, sc, inv, BITS, q);
    if (BITS == 8) {
      uint2 out;
      out.x = pack4_bytes(q[0], q[1], q[2], q[3]);
      out.y = pack4_bytes(q[4], q[5], q[6], q[7]);
      *reinterpret_cast<uint2*>(bcodes + e) = out;
    } else {
      uint32_t out = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) out |= (uint32_t)((q[i] + 8) & 0xF) << (4 * i);
      *reinterpret_cast<uint32_t*>(bcodes + (e >> 1)) = out;
    }
  }
}

// ---- per-tensor fast path (one scale for the whole array, n % 8 == 0): vectorised absmax with one atomicMax per CTA,
// then a vectorised apply; both HBM-bound (read 2x, write once).
template <typename T>
__global__ void __launch_bounds__(256) absmax_flat_kernel(const T* __restrict__ src, unsigned int* __restrict__ amax_bits,
                                                          uint64_t n8) {
  __shared__ float red[8];
  float amax = 0.f;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (uint64_t)gridDim.x * blockDim.x) {
    float x[8];
    Vec8<T>::load(src + i * 8, x);
#pragma unroll
    for (int k = 0; k < 8; ++k) amax = fmaxf(amax, fabsf(x[k]));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = amax;
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 1; i < 8; ++i) amax = fmaxf(amax, red[i]);
    atomicMax(amax_bits, __float_as_uint(amax));
  }
}

template <typename T, int BITS>
__global__ void __launch_bounds__(256) quant_flat_kernel(const T* __restrict__ src, uint8_t* __restrict__ codes,
                                                         const float* __restrict__ scale, uint64_t n8) {
  const float sc = *scale;
  const float inv = inv_scale(sc);
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (uint64_t)gridDim.x * blockDim.x) {
    float x[8];
    Vec8<T>::load(src + i * 8, x);
    int q[8];
    quant_codes8(x, sc, inv, BITS, q);
    if (BITS == 8) {
      uint2 out;
      out.x = pack4_bytes(q[0], q[1], q[2], q[3]);
      out.y = pack4_bytes(q[4], q[5], q[6], q[7]);
      reinterpret_cast<uint2*>(codes)[i] = out;
    } else {
      uint32_t out = 0;
#pragma unroll
      for (int k = 0; k < 8; ++k) out |= (uint32_t)((q[k] + 8) & 0xF) << (4 * k);
      reinterpret_cast<uint32_t*>(codes)[i] = out;
    }
  }
}

// ---- generic path, kernel 1: absmax of arbitrary block_rows x block_cols tiles via uint-bit atomicMax
// (|x| >= 0, so the IEEE bit pattern orders like the value -- the reference GPU path does the same,
// GEMMRuntimeQuantization.swift:22-41).
template <typename T>
__global__ void absmax_generic_kernel(const T* __restrict__ src, unsigned int* __restrict__ amax_bits, uint64_t rows,
                                      uint64_t cols, uint32_t block_rows, uint32_t block_cols, uint64_t group_rows,
                                      uint32_t nb_per_group, uint32_t nbc) {
  const uint64_t n = rows * cols;
  uint64_t cur_blk = ~0ull;
  float cur = 0.f;
  // each thread walks a contiguous chunk so consecutive elements mostly share a block -> few atomics
  const uint64_t chunk = 64;
  for (uint64_t base = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * chunk; base < n;
       base += (uint64_t)gridDim.x * blockDim.x * chunk) {
    uint64_t end = base + chunk < n ? base + chunk : n;
    for (uint64_t e = base; e < end; ++e) {
      uint64_t r = e / cols, c = e - r * cols;
      uint64_t g = r / group_rows;
      uint64_t blk = (g * nb_per_group + (r - g * group_rows) / block_rows) * nbc + c / block_cols;
      if (blk != cur_blk) {
        if (cur_blk != ~0ull) atomicMax(amax_bits + cur_blk, __float_as_uint(cur));
        cur_blk = blk; cur = 0.f;
      }
      cur = fmaxf(cur, fabsf(to_f32<T>(src[e])));
    }
  }
  if (cur_blk != ~0ull) atomicMax(amax_bits + cur_blk, __float_as_uint(cur));
}

__global__ void finalize_scales_kernel(float* scales /* in: absmax bits, out: scale */, uint64_t nblocks, int bits,
                                       float floor_v) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nblocks) scales[i] = make_scale(scales[i], bits, floor_v);
}

// ---- generic path, kernel 2: one thread per output byte pair
template <typename T, int BITS>
__global__ void quant_apply_generic_kernel(const T* __restrict__ src, uint8_t* __restrict__ codes,
                                           const float* __restrict__ scales, uint64_t rows, uint64_t cols,
                                           uint32_t block_rows, uint32_t block_cols, uint64_t group_rows,
                                           uint32_t nb_per_group, uint32_t nbc) {
  const uint64_t n = rows * cols;
  for (uint64_t e = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 2; e < n;
       e += (uint64_t)gridDim.x * blockDim.x * 2) {
    int q[2] = {0, 0};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      uint64_t ee = e + i;
      if (ee >= n) break;
      uint64_t r = ee / cols, c = ee - r * cols;
      uint64_t g = r / group_rows;
      uint64_t blk = (g * nb_per_group + (r - g * group_rows) / block_rows) * nbc + c / block_cols;
      q[i] = quant_code(to_f32<T>(src[ee]), scales[blk], BITS);
    }
    if (BITS == 8) {
      codes[e] = (uint8_t)(q[0] & 0xFF);
      if (e + 1 < n) codes[e + 1] = (uint8_t)(q[1] & 0xFF);
    } else {
      codes[e >> 1] = (uint8_t)(((q[0] + 8) & 0xF) | (((q[1] + 8) & 0xF) << 4));
    }
  }
}

template <int BITS>
__global__ void dequant_kernel(const uint8_t* __restrict__ codes, const float* __restrict__ scales,
                               float* __restrict__ out, uint64_t rows, uint64_t cols, uint32_t block_rows,
                               uint32_t block_cols, uint32_t nbc) {
  const uint64_t n = rows * cols;
  for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t r = e / cols, c = e - r * cols;
    float sc = scales[(r / block_rows) * nbc + c / block_cols];
    int q;
    if (BITS == 8) q = reinterpret_cast<const int8_t*>(codes)[e];
    else { uint8_t b = codes[e >> 1]; q = (int)((e & 1) ? (b >> 4) : (b & 0xF)) - 8; }
    out[e] = (float)q * sc;
  }
}

// ---- operands of the tensor-core backward of quantised attention: the values the reference's backward sees (dequantised
// codes, QuantizedAttention.swift:1428-1608 / MFABridge+Quantized.swift:365-533) as bf16, 16 elements per thread.  Scales:
// one per tensor (by value or scales[0]) or one per block of `block_rows` tokens inside each (b, head) of rows_per_head rows.
template <int BITS>
__global__ void dequant_bf16_kernel(const uint8_t* __restrict__ codes, __nv_bfloat16* __restrict__ out,
                                    const float* __restrict__ scales, float one_scale, int zero_point, int block_rows,
                                    int nb_per_head, uint64_t rows_per_head, uint32_t D, uint64_t n16) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t row = (i * 16) / D;
    float sc = one_scale;
    if (scales) {
      const uint64_t hd = row / rows_per_head;
      sc = nb_per_head > 0 ? scales[hd * nb_per_head + (row - hd * rows_per_head) / block_rows] : scales[0];
    }
    int q[16];
    if (BITS == 8) {
      const int4 v = reinterpret_cast<const int4*>(codes)[i];
      const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 16; ++k) q[k] = (int)(int8_t)((w[k >> 2] >> (8 * (k & 3))) & 0xff);
    } else {
      const uint2 v = reinterpret_cast<const uint2*>(codes)[i];
      const uint32_t w[2] = {v.x, v.y};
#pragma unroll
      for (int k = 0; k < 16; ++k) q[k] = (int)((w[k >> 3] >> (4 * (k & 7))) & 0xf) - 8;
    }
    uint32_t o[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const __nv_bfloat162 h = __floats2bfloat162_rn((float)(q[2 * k] - zero_point) * sc, (float)(q[2 * k + 1] - zero_point) * sc);
      o[k] = *reinterpret_cast<const uint32_t*>(&h);
    }
    reinterpret_cast<uint4*>(out)[2 * i] = make_uint4(o[0], o[1], o[2], o[3]);
    reinterpret_cast<uint4*>(out)[2 * i + 1] = make_uint4(o[4], o[5], o[6], o[7]);
  }
}

// fp32 / fp16 -> bf16 (the upstream gradient of the same backward), 8 elements per thread
template <typename T>
__global__ void to_bf16_kernel(const T* __restrict__ src, __nv_bfloat16* __restrict__ out, uint64_t n8) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(to_f32<T>(src[8 * i + 2 * k]), to_f32<T>(src[8 * i + 2 * k + 1]));
      o[k] = *reinterpret_cast<const uint32_t*>(&h);
    }
    reinterpret_cast<uint4*>(out)[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// ---- merge of two attention partials over disjoint key sets (log2-domain L, SURVEY 8e)
__global__ void merge_partials_kernel(float* __restrict__ o_acc, float* __restrict__ l_acc,
                                      const float* __restrict__ o_part, const float* __restrict__ l_part,
                                      uint64_t rows, uint32_t D) {
  const uint64_t row = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float la = l_acc[row], lp = l_part[row];
  if (lp == -CUDART_INF_F) return;
  const float m = fmaxf(la, lp);
  const float wa = lse_merge_weight(la, m), wp = lse_merge_weight(lp, m);
  const float s = wa + wp;
  const float ca = wa / s, cp = wp / s;
  float* oa = o_acc + row * D;
  const float* op = o_part + row * D;
  if ((D & 3) == 0) {
    for (uint32_t d = lane * 4; d < D; d += 128) {
      float4 a = *reinterpret_cast<float4*>(oa + d);
      const float4 b = *reinterpret_cast<const float4*>(op + d);
      a.x = a.x * ca + b.x * cp; a.y = a.y * ca + b.y * cp; a.z = a.z * ca + b.z * cp; a.w = a.w * ca + b.w * cp;
      *reinterpret_cast<float4*>(oa + d) = a;
    }
  } else {
    for (uint32_t d = lane; d < D; d += 32) oa[d] = oa[d] * ca + op[d] * cp;
  }
  __syncwarp();
  if (lane == 0) l_acc[row] = lse_merge_total(m, s);
}

// ---- in-place FWHT over blocks of n = 2^k <= 1024 fp32 values, scaled by 1/sqrt(n)
// (metal-flash-attention/Sources/FlashAttention/Attention/HadamardRotation.swift:113-147 does this with one
// thread per block; here a CTA of n/2 butterflies per stage, data staged in shared memory).
__global__ void hadamard_kernel(float* __restrict__ data, uint32_t n, uint32_t num_blocks) {
  extern __shared__ float buf[];
  for (uint32_t blk = blockIdx.x; blk < num_blocks; blk += gridDim.x) {
    float* p = data + (uint64_t)blk * n;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) buf[i] = p[i];
    __syncthreads();
    for (uint32_t h = 1; h < n; h <<= 1) {
      for (uint32_t t = threadIdx.x; t < n / 2; t += blockDim.x) {
        uint32_t i = ((t / h) * 2 * h) + (t % h);
        float a = buf[i], b = buf[i + h];
        buf[i] = a + b; buf[i + h] = a - b;
      }
      __syncthreads();
    }
    const float norm = rsqrtf((float)n);
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) p[i] = buf[i] * norm;
    __syncthreads();
  }
}

// ---- interleaved-pair RoPE (Sources/MFABridge/MFABridge.swift:269-319): (x0, x1) -> (x0 c - x1 s, x0 s + x1 c) (rope_pair).
// Tables follow the reference contract exactly: pair-duplicated fp32 [S, D] (only the even entry of a pair is read),
// element t = b * table_batch_stride + s * D + 2 * pair, table_batch_stride = 0 (shared) or S * D ([B, S, D]).
template <typename T> __device__ __forceinline__ T from_f32(float x);
template <> __device__ __forceinline__ float from_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ __half from_f32<__half>(float x) { return __float2half_rn(x); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }

template <typename T>
__global__ void rope_kernel(const T* __restrict__ src, T* __restrict__ dst, const float* __restrict__ cos_t,
                            const float* __restrict__ sin_t, int64_t sB, int64_t sH, int64_t sS,
                            int64_t table_batch_stride, bool negate_sin, uint32_t B, uint32_t H, uint32_t S, uint32_t D) {
  const uint32_t half = D / 2;
  const uint64_t total = (uint64_t)B * H * S * half;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t j = (uint32_t)(i % half);
    uint64_t t = i / half;
    uint32_t s = (uint32_t)(t % S); t /= S;
    uint32_t h = (uint32_t)(t % H);
    uint32_t b = (uint32_t)(t / H);
    const int64_t in = b * sB + h * sH + s * sS + 2 * j;
    const int64_t out = (((int64_t)b * H + h) * S + s) * D + 2 * j;     // dst is contiguous BHSD
    const int64_t ti = b * table_batch_stride + (int64_t)s * D + 2 * j;
    float c = cos_t[ti], sn = sin_t[ti];
    if (negate_sin) sn = -sn;
    float y0, y1;
    rope_pair(to_f32<T>(src[in]), to_f32<T>(src[in + 1]), c, sn, y0, y1);
    dst[out] = from_f32<T>(y0);
    dst[out + 1] = from_f32<T>(y1);
  }
}

template <typename T>
__global__ void convert_kernel(const float* __restrict__ src, T* __restrict__ dst, uint64_t n) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
    dst[i] = from_f32<T>(src[i]);
}

inline unsigned grid_for(uint64_t work_items, int threads) {
  uint64_t g = (work_items + threads - 1) / threads;
  const uint64_t cap = 148ull * 32;
  return (unsigned)(g < 1 ? 1 : (g > cap ? cap : g));
}

template <typename T>
cudaError_t quantize_typed(const T* src, uint8_t* codes, float* scales, uint64_t rows, uint64_t cols, uint32_t br,
                           uint32_t bc, uint64_t group_rows, int bits, float floor_v, cudaStream_t st) {
  const uint32_t nb_per_group = (uint32_t)((group_rows + br - 1) / br);
  const uint64_t ngroups = (rows + group_rows - 1) / group_rows;
  const uint32_t nbc = (uint32_t)((cols + bc - 1) / bc);
  const uint64_t nblocks = ngroups * nb_per_group * nbc;
  const uint64_t span = (uint64_t)br * cols;
  const bool aligned = (cols % 8 == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0) &&
                       ((reinterpret_cast<uintptr_t>(codes) & 7) == 0);
  if (bc == cols && aligned && span <= 65536) {
    if (span <= 2048) {
      unsigned grid = (unsigned)((nblocks + 7) / 8);
      if (bits == 8) quant_span_kernel<T, 8, true><<<grid, 256, 0, st>>>(src, codes, scales, rows, cols, br, group_rows, nb_per_group, nblocks, floor_v);
      else quant_span_kernel<T, 4, true><<<grid, 256, 0, st>>>(src, codes, scales, rows, cols, br, group_rows, nb_per_group, nblocks, floor_v);
    } else {
      unsigned grid = (unsigned)nblocks;
      // CTA size: with 256 threads ~6 CTAs fit an SM (888 on the chip), so the 1728 blocks of a FLUX tensor run as two waves;
      // 128-thread CTAs (13 per SM) hold them all at once -- and measure SLOWER, 20.3 against 18.2 us under ncu
      // (profiles/r02bo_helpers_{128,256}.csv): the wave count is not what bounds this pass either.
      if (bits == 8) quant_span_kernel<T, 8, false><<<grid, 256, 0, st>>>(src, codes, scales, rows, cols, br, group_rows, nb_per_group, nblocks, floor_v);
      else quant_span_kernel<T, 4, false><<<grid, 256, 0, st>>>(src, codes, scales, rows, cols, br, group_rows, nb_per_group, nblocks, floor_v);
    }
    ++g_launch_count;
    g_last_kernel = "quant_span";
    return cudaGetLastError();
  }
  // generic: absmax (atomics) -> scales -> apply
  cudaError_t e = cudaMemsetAsync(scales, 0, nblocks * sizeof(float), st);
  if (e != cudaSuccess) return e;
  const uint64_t n = rows * cols;
  if (nblocks == 1 && (n % 8) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(codes) & 7) == 0) {
    const unsigned grid = grid_for(n / 8, 256) < 148u * 8 ? grid_for(n / 8, 256) : 148u * 8;
    absmax_flat_kernel<T><<<grid, 256, 0, st>>>(src, reinterpret_cast<unsigned int*>(scales), n / 8);
    finalize_scales_kernel<<<1, 32, 0, st>>>(scales, 1, bits, floor_v);
    if (bits == 8) quant_flat_kernel<T, 8><<<grid, 256, 0, st>>>(src, codes, scales, n / 8);
    else quant_flat_kernel<T, 4><<<grid, 256, 0, st>>>(src, codes, scales, n / 8);
    g_launch_count += 3;
    g_last_kernel = "quant_flat";
    return cudaGetLastError();
  }
  absmax_generic_kernel<T><<<grid_for((n + 63) / 64, 256), 256, 0, st>>>(
      src, reinterpret_cast<unsigned int*>(scales), rows, cols, br, bc, group_rows, nb_per_group, nbc);
  finalize_scales_kernel<<<(unsigned)((nblocks + 255) / 256), 256, 0, st>>>(scales, nblocks, bits, floor_v);
  if (bits == 8) quant_apply_generic_kernel<T, 8><<<grid_for((n + 1) / 2, 256), 256, 0, st>>>(src, codes, scales, rows, cols, br, bc, group_rows, nb_per_group, nbc);
  else quant_apply_generic_kernel<T, 4><<<grid_for((n + 1) / 2, 256), 256, 0, st>>>(src, codes, scales, rows, cols, br, bc, group_rows, nb_per_group, nbc);
  g_launch_count += 3;
  g_last_kernel = "quant_generic";
  return cudaGetLastError();
}

}  // namespace

// group_rows: quantisation blocks restart every group_rows rows (one (batch, head) slab); 0 = no grouping.
cudaError_t launch_quantize_grouped(const void* src, int src_dtype, void* codes, float* scales, uint64_t rows,
                                    uint64_t cols, uint32_t block_rows, uint32_t block_cols, uint64_t group_rows,
                                    int bits, float scale_floor, cudaStream_t st) {
  if (rows == 0 || cols == 0) return cudaSuccess;
  if (bits != 8 && bits != 4) return cudaErrorInvalidValue;
  if (group_rows == 0 || group_rows > rows) group_rows = rows;
  uint32_t br = (block_rows == 0 || block_rows > group_rows) ? (uint32_t)group_rows : block_rows;
  uint32_t bc = (block_cols == 0 || block_cols > cols) ? (uint32_t)cols : block_cols;
  if (bits == 4 && bc != cols && ((bc & 1) || (cols & 1))) return cudaErrorInvalidValue;  // nibble pairs must share a block row
  uint8_t* c8 = reinterpret_cast<uint8_t*>(codes);
  switch (src_dtype) {
    case kF32: return quantize_typed(reinterpret_cast<const float*>(src), c8, scales, rows, cols, br, bc, group_rows, bits, scale_floor, st);
    case kF16: return quantize_typed(reinterpret_cast<const __half*>(src), c8, scales, rows, cols, br, bc, group_rows, bits, scale_floor, st);
    case kBF16: return quantize_typed(reinterpret_cast<const __nv_bfloat16*>(src), c8, scales, rows, cols, br, bc, group_rows, bits, scale_floor, st);
    default: return cudaErrorInvalidValue;
  }
}

cudaError_t launch_quantize(const void* src, int src_dtype, void* codes, float* scales, uint64_t rows, uint64_t cols,
                            uint32_t block_rows, uint32_t block_cols, int bits, float scale_floor, cudaStream_t st) {
  return launch_quantize_grouped(src, src_dtype, codes, scales, rows, cols, block_rows, block_cols, 0, bits, scale_floor, st);
}

cudaError_t launch_dequantize(const void* codes, const float* scales, float* out, uint64_t rows, uint64_t cols,
                              uint32_t block_rows, uint32_t block_cols, int bits, cudaStream_t st) {
  if (rows == 0 || cols == 0) return cudaSuccess;
  uint32_t br = (block_rows == 0 || block_rows > rows) ? (uint32_t)rows : block_rows;
  uint32_t bc = (block_cols == 0 || block_cols > cols) ? (uint32_t)cols : block_cols;
  uint32_t nbc = (uint32_t)((cols + bc - 1) / bc);
  unsigned grid = grid_for(rows * cols, 256);
  if (bits == 8) dequant_kernel<8><<<grid, 256, 0, st>>>(reinterpret_cast<const uint8_t*>(codes), scales, out, rows, cols, br, bc, nbc);
  else if (bits == 4) dequant_kernel<4><<<grid, 256, 0, st>>>(reinterpret_cast<const uint8_t*>(codes), scales, out, rows, cols, br, bc, nbc);
  else return cudaErrorInvalidValue;
  ++g_launch_count;
  return cudaGetLastError();
}

cudaError_t launch_dequantize_bf16(const void* codes, int bits, const QuantView& q, void* out, uint64_t heads,
                                   uint64_t rows_per_head, uint32_t D, cudaStream_t st) {
  const uint64_t n = heads * rows_per_head * D;
  if (n == 0) return cudaSuccess;
  if ((n % 16) || (D % 16)) return cudaErrorInvalidValue;
  const bool blocks = q.scales && q.block_rows > 0;
  const int nb = blocks ? (int)((rows_per_head + q.block_rows - 1) / q.block_rows) : 0;
  const unsigned grid = grid_for(n / 16, 256);
  if (bits == 8)
    dequant_bf16_kernel<8><<<grid, 256, 0, st>>>(reinterpret_cast<const uint8_t*>(codes), reinterpret_cast<__nv_bfloat16*>(out),
                                                q.scales, q.scale, q.zero_point, blocks ? q.block_rows : 1, nb, rows_per_head, D, n / 16);
  else if (bits == 4)
    dequant_bf16_kernel<4><<<grid, 256, 0, st>>>(reinterpret_cast<const uint8_t*>(codes), reinterpret_cast<__nv_bfloat16*>(out),
                                                q.scales, q.scale, q.zero_point, blocks ? q.block_rows : 1, nb, rows_per_head, D, n / 16);
  else return cudaErrorInvalidValue;
  ++g_launch_count;
  return cudaGetLastError();
}

cudaError_t launch_to_bf16(const void* src, int src_dtype, void* out, uint64_t n, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  if (n % 8) return cudaErrorInvalidValue;
  const unsigned grid = grid_for(n / 8, 256);
  if (src_dtype == kF32) to_bf16_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(src), reinterpret_cast<__nv_bfloat16*>(out), n / 8);
  else if (src_dtype == kF16) to_bf16_kernel<__half><<<grid, 256, 0, st>>>(reinterpret_cast<const __half*>(src), reinterpret_cast<__nv_bfloat16*>(out), n / 8);
  else return cudaErrorInvalidValue;
  ++g_launch_count;
  return cudaGetLastError();
}

cudaError_t launch_merge_partials(float* o_acc, float* l_acc, const float* o_part, const float* l_part, uint64_t rows,
                                  uint32_t D, cudaStream_t st) {
  if (rows == 0) return cudaSuccess;
  merge_partials_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(o_acc, l_acc, o_part, l_part, rows, D);
  ++g_launch_count;
  return cudaGetLastError();
}

// Blocks of n = 32 E values, E = 1 .. 32: one warp per block, lane L holds elements [E L, E L + E) in registers (vector loads:
// a warp request covers the whole block, fully coalesced), the butterflies with span h < E stay inside the lane, those with
// h >= E exchange with lane L ^ (h / E) by shuffle -- no shared memory, no barriers; HBM-bound (4 B in + 4 B out per element).
// The shared-memory kernel above (one CTA per block, a barrier per stage) moved a 512-byte head_dim-128 block per CTA.
template <int E>
__global__ void __launch_bounds__(256) hadamard_warp_kernel(float* __restrict__ data, uint32_t num_blocks) {
  const uint32_t lane = threadIdx.x & 31;
  const float norm = rsqrtf((float)(32 * E));
  for (uint64_t blk = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5); blk < num_blocks; blk += (uint64_t)gridDim.x * 8) {
    float* p = data + blk * (32 * E) + lane * E;
    float x[E];
    if constexpr (E >= 4) {
#pragma unroll
      for (int i = 0; i < E / 4; ++i) {
        const float4 v = reinterpret_cast<const float4*>(p)[i];
        x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
      }
    } else if constexpr (E == 2) {
      const float2 v = *reinterpret_cast<const float2*>(p);
      x[0] = v.x; x[1] = v.y;
    } else {
      x[0] = p[0];
    }
#pragma unroll
    for (int h = 1; h < E; h <<= 1) {
#pragma unroll
      for (int i = 0; i < E; ++i) {
        if ((i & h) == 0) {
          const float a = x[i], b = x[i + h];
          x[i] = a + b; x[i + h] = a - b;
        }
      }
    }
#pragma unroll
    for (int m = 1; m < 32; m <<= 1) {
      const bool upper = (lane & m) != 0;
#pragma unroll
      for (int i = 0; i < E; ++i) {
        const float v = __shfl_xor_sync(0xffffffffu, x[i], m);
        x[i] = upper ? v - x[i] : x[i] + v;
      }
    }
    if constexpr (E >= 4) {
#pragma unroll
      for (int i = 0; i < E / 4; ++i)
        reinterpret_cast<float4*>(p)[i] = make_float4(x[4 * i] * norm, x[4 * i + 1] * norm, x[4 * i + 2] * norm, x[4 * i + 3] * norm);
    } else if constexpr (E == 2) {
      *reinterpret_cast<float2*>(p) = make_float2(x[0] * norm, x[1] * norm);
    } else {
      p[0] = x[0] * norm;
    }
  }
}

template <int E>
void launch_hadamard_warp(float* data, uint32_t num_blocks, cudaStream_t st) {
  const unsigned want = (num_blocks + 7) / 8, cap = 148u * 8 * 4;
  hadamard_warp_kernel<E><<<want < cap ? want : cap, 256, 0, st>>>(data, num_blocks);
}

cudaError_t launch_hadamard(float* data, uint32_t block_size, uint32_t num_blocks, cudaStream_t st) {
  if (block_size == 0 || block_size > 1024 || (block_size & (block_size - 1))) return cudaErrorInvalidValue;
  if (num_blocks == 0) return cudaSuccess;
  if (block_size >= 32 && (reinterpret_cast<uintptr_t>(data) & 15) == 0) {
    switch (block_size / 32) {
      case 1: launch_hadamard_warp<1>(data, num_blocks, st); break;
      case 2: launch_hadamard_warp<2>(data, num_blocks, st); break;
      case 4: launch_hadamard_warp<4>(data, num_blocks, st); break;
      case 8: launch_hadamard_warp<8>(data, num_blocks, st); break;
      case 16: launch_hadamard_warp<16>(data, num_blocks, st); break;
      default: launch_hadamard_warp<32>(data, num_blocks, st); break;
    }
    ++g_launch_count;
    return cudaGetLastError();
  }
  unsigned threads = block_size / 2 < 32 ? 32 : block_size / 2;
  unsigned grid = num_blocks < 148u * 16 ? num_blocks : 148u * 16;
  hadamard_kernel<<<grid, threads, block_size * sizeof(float), st>>>(data, block_size, num_blocks);
  ++g_launch_count;
  return cudaGetLastError();
}

cudaError_t launch_rope(const void* src, void* dst, const float* cos_t, const float* sin_t, int64_t sB, int64_t sH,
                        int64_t sS, int64_t table_batch_stride, bool negate_sin, uint32_t B, uint32_t H, uint32_t S,
                        uint32_t D, int dtype, cudaStream_t st) {
  if (D & 1) return cudaErrorInvalidValue;
  uint64_t total = (uint64_t)B * H * S * (D / 2);
  if (total == 0) return cudaSuccess;
  unsigned grid = grid_for(total, 256);
  switch (dtype) {
    case kF32: rope_kernel<float><<<grid, 256, 0, st>>>((const float*)src, (float*)dst, cos_t, sin_t, sB, sH, sS, table_batch_stride, negate_sin, B, H, S, D); break;
    case kF16: rope_kernel<__half><<<grid, 256, 0, st>>>((const __half*)src, (__half*)dst, cos_t, sin_t, sB, sH, sS, table_batch_stride, negate_sin, B, H, S, D); break;
    case kBF16: rope_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)src, (__nv_bfloat16*)dst, cos_t, sin_t, sB, sH, sS, table_batch_stride, negate_sin, B, H, S, D); break;
    default: return cudaErrorInvalidValue;
  }
  ++g_launch_count;
  return cudaGetLastError();
}

cudaError_t launch_convert_from_f32(const float* src, void* dst, int dst_dtype, uint64_t n, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  unsigned grid = grid_for(n, 256);
  if (dst_dtype == kF16) convert_kernel<__half><<<grid, 256, 0, st>>>(src, (__half*)dst, n);
  else if (dst_dtype == kBF16) convert_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(src, (__nv_bfloat16*)dst, n);
  else return cudaErrorInvalidValue;
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace mfa
