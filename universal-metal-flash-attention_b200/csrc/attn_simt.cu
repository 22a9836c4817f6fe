// attn_simt.cu -- exact-fp32 SIMT attention kernels (forward, D-term, dQ, dK/dV).
//
// This is the path for fp32 inputs (1e-5 parity needs real fp32 FMAs; tensor cores only offer TF32), for head
// dimensions / layouts the tcgen05 kernels do not cover (D not in {64,128}, transposed operands, GQA,
// dequantise-on-load int8/int4 operands) and for the backward pass until the tcgen05 backward lands.
// Math follows the reference kernel loops (metal-flash-attention/Sources/FlashAttention/Attention/
// AttentionKernel/AttentionKernel+Source.swift:372-511, +Softmax.swift:641-802) re-derived for CUDA:
//   forward      m' = max(m, rowmax(z)), P = exp2(z - m'), l = l*2^(m-m') + rowsum(P), O = O*2^(m-m') + P V
//                with z = log2e * (scale * q.k + mask); L = m + log2(l)
//   backwardQ    P = exp2(z - L), dP = dO V^T, dS = P * (scale*dP - Dterm), dQ += dS K        (Dterm = scale*sum dO*O)
//   backwardKV   dV += P^T dO, dK += dS^T Q
// Tiles: 32 "outer" rows per CTA (resident in smem), 32 "inner" rows per step, 256 threads.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math_constants.h>

#include "common.h"

namespace mfa {

unsigned long long g_launch_count = 0;
const char* g_last_kernel = "none";

namespace {

constexpr int TR = 32;        // outer rows per CTA
constexpr int TC = 32;        // inner rows per step
constexpr int NT = 256;       // threads per CTA
constexpr int MAXD = 256;
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ float load_elem(const void* base, int dtype, int64_t idx) {
  switch (dtype) {
    case kF32: return reinterpret_cast<const float*>(base)[idx];
    case kF16: return __half2float(reinterpret_cast<const __half*>(base)[idx]);
    case kBF16: return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[idx]);
    case kI8: return (float)reinterpret_cast<const int8_t*>(base)[idx];
    default: {  // kI4: two codes per byte, even element in the low nibble, stored +8
      uint8_t b = reinterpret_cast<const uint8_t*>(base)[idx >> 1];
      return (float)((int)((idx & 1) ? (b >> 4) : (b & 0xF)) - 8);
    }
  }
}

__device__ __forceinline__ float mask_value(const AttnParams& p, int b, int h, int r, int c) {
  if (p.mask_kind == kMaskNone) return 0.f;
  int64_t idx = b * p.mask_sb + h * p.mask_sh + r * p.mask_sq + c * p.mask_sk;
  if (p.mask_kind == kMaskBool) {
    return reinterpret_cast<const uint8_t*>(p.mask)[idx] ? 0.f : -CUDART_INF_F;
  }
  switch (p.mask_scalar) {
    case kMaskF16: return __half2float(reinterpret_cast<const __half*>(p.mask)[idx]);
    case kMaskBF16: return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.mask)[idx]);
    default: return reinterpret_cast<const float*>(p.mask)[idx];
  }
}

// Load rows [row0, row0+nrows) x D of a [.,.,S,D] view into smem tile[nrows][ld] as fp32 (zero padded to Dp
// columns and past `S`).  Applies dequantisation for int8/int4 operands; scale_base = index of the first block
// scale of this (batch, head).
__device__ void load_tile(float* tile, int ld, const TensorView& t, int dtype, const QuantView& qv, int b, int h,
                          int64_t scale_base, int row0, int nrows, int S, int D, int Dp) {
  const int64_t base = b * t.sb + h * t.sh;
  for (int i = threadIdx.x; i < nrows * Dp; i += NT) {
    int r = i / Dp, d = i - r * Dp;
    int s = row0 + r;
    float x = 0.f;
    if (s < S && d < D) {
      x = load_elem(t.ptr, dtype, base + s * t.ss + d * t.sd);
      if (dtype == kI8 || dtype == kI4) {
        float sc = qv.scales ? (qv.block_rows > 0 ? qv.scales[scale_base + s / qv.block_rows] : qv.scales[0])
                             : qv.scale;
        x = (x - (float)qv.zero_point) * sc;
      }
    }
    tile[r * ld + d] = x;
  }
}

// S[TR][TC] = A[TR][D] . B[TC][D]^T ; thread (ty,tx) computes rows ty*4..ty*4+3, column tx.
__device__ __forceinline__ void tile_abt(const float* A, const float* Bm, int ld, int Dp, float out[4]) {
  const int ty = threadIdx.x >> 5, tx = threadIdx.x & 31;
  const float* a0 = A + (ty * 4) * ld;
  const float* b0 = Bm + tx * ld;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll 4
  for (int d = 0; d < Dp; ++d) {
    float bv = b0[d];
    s0 = fmaf(a0[d], bv, s0);
    s1 = fmaf(a0[ld + d], bv, s1);
    s2 = fmaf(a0[2 * ld + d], bv, s2);
    s3 = fmaf(a0[3 * ld + d], bv, s3);
  }
  out[0] = s0; out[1] = s1; out[2] = s2; out[3] = s3;
}

// acc[4][8] += W[TR][TC] (rows ty*4.., stored with stride ldw; transposed read if TRANS) . Bm[TC][D]
// thread owns rows ty*4..+3 and columns tx + 32*i.
template <bool TRANS>
__device__ __forceinline__ void tile_acc(const float* W, int ldw, const float* Bm, int ld, int Dp, float acc[4][8]) {
  const int ty = threadIdx.x >> 5, tx = threadIdx.x & 31;
  const int ng = Dp >> 5;
  for (int c = 0; c < TC; ++c) {
    float w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = TRANS ? W[c * ldw + ty * 4 + j] : W[(ty * 4 + j) * ldw + c];
    const float* br = Bm + c * ld + tx;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i < ng) {
        float bv = br[i * 32];
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[j][i] = fmaf(w[j], bv, acc[j][i]);
      }
    }
  }
}

__device__ __forceinline__ void store_out(void* base, int dtype, int64_t idx, float x) {
  if (dtype == kF32) reinterpret_cast<float*>(base)[idx] = x;
  else if (dtype == kF16) reinterpret_cast<__half*>(base)[idx] = __float2half_rn(x);
  else reinterpret_cast<__nv_bfloat16*>(base)[idx] = __float2bfloat16_rn(x);
}

// z (log2 domain) for element (row r, key c) from the raw dot product; `visible` comes from the causal / window / segment rule
// (row_key_range / key_query_range).
__device__ __forceinline__ float logit(const AttnParams& p, int b, int h, int r, int c, float dot, bool visible) {
  if (!visible || r >= p.Sq || c >= p.Skv) return -CUDART_INF_F;
  float z = dot * p.scale;
  if (p.mask_kind != kMaskNone) z += mask_value(p, b, h, r, c);
  return z * kLog2e;
}

// ------------------------------------------------------------------------------------------- forward
__global__ void __launch_bounds__(NT) fwd_simt_kernel(AttnParams p) {
  extern __shared__ float smem[];
  const int Dp = (p.D + 31) & ~31, ld = Dp + 1;
  float* Qs = smem;                    // [TR][ld]
  float* Ks = Qs + TR * ld;            // [TC][ld]
  float* Vs = Ks + TC * ld;            // [TC][ld]
  float* Ss = Vs + TC * ld;            // [TR][TC+1]
  float* row_m = Ss + TR * (TC + 1);   // [TR]
  float* row_l = row_m + TR;           // [TR]
  float* row_c = row_l + TR;           // [TR] correction factor for this step

  const int b = blockIdx.z, h = blockIdx.y, r0 = blockIdx.x * TR;
  const int hk = h / (p.H / p.Hkv);
  const int ty = threadIdx.x >> 5, tx = threadIdx.x & 31;
  const int nbq = p.qq.block_rows > 0 ? (p.Sq + p.qq.block_rows - 1) / p.qq.block_rows : 1;
  const int nbk = p.qk.block_rows > 0 ? (p.Skv + p.qk.block_rows - 1) / p.qk.block_rows : 1;
  const int nbv = p.qv.block_rows > 0 ? (p.Skv + p.qv.block_rows - 1) / p.qv.block_rows : 1;

  const int64_t sbq = ((int64_t)b * p.H + h) * nbq, sbk = ((int64_t)b * p.Hkv + hk) * nbk, sbv = ((int64_t)b * p.Hkv + hk) * nbv;
  load_tile(Qs, ld, p.q, p.in_dtype, p.qq, b, h, sbq, r0, TR, p.Sq, p.D, Dp);
  if (threadIdx.x < TR) { row_m[threadIdx.x] = -CUDART_INF_F; row_l[threadIdx.x] = 0.f; }
  float acc[4][8];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[j][i] = 0.f;

  __shared__ int rlo[TR], rhi[TR];      // visible keys of each row
  if (threadIdx.x < TR) row_key_range(p.causal, p.window, p.Sq, p.Skv, p.cu_q, p.cu_k, p.nseq, r0 + threadIdx.x, rlo[threadIdx.x], rhi[threadIdx.x]);
  int klo, khi;
  block_key_range(p.causal, p.window, p.Sq, p.Skv, p.cu_q, p.cu_k, p.nseq, r0, min(r0 + TR, p.Sq), klo, khi);
  klo = (klo / TC) * TC;
  for (int c0 = klo; c0 < khi; c0 += TC) {
    __syncthreads();
    load_tile(Ks, ld, p.k, p.in_dtype, p.qk, b, hk, sbk, c0, TC, p.Skv, p.D, Dp);
    load_tile(Vs, ld, p.v, p.in_dtype, p.qv, b, hk, sbv, c0, TC, p.Skv, p.D, Dp);
    __syncthreads();
    float s[4];
    tile_abt(Qs, Ks, ld, Dp, s);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int r = ty * 4 + j;
      float z = logit(p, b, h, r0 + r, c0 + tx, s[j], c0 + tx >= rlo[r] && c0 + tx < rhi[r]);
      // row max across the warp (all 32 lanes share row r)
      float mx = z;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float m_old = row_m[r];
      float m_new = fmaxf(m_old, mx);
      float m_safe = (m_new == -CUDART_INF_F) ? 0.f : m_new;
      float pv = exp2f(z - m_safe);                  // z = -inf -> 0
      float sum = pv;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      float corr = exp2f(m_old - m_safe);            // m_old = -inf -> 0
      Ss[r * (TC + 1) + tx] = pv;
      __syncwarp();
      if (tx == 0) { row_m[r] = m_new; row_l[r] = row_l[r] * corr + sum; row_c[r] = corr; }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float cf = row_c[ty * 4 + j];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[j][i] *= cf;
    }
    tile_acc<false>(Ss, TC + 1, Vs, ld, Dp, acc);
  }
  __syncthreads();
  const int64_t obase = b * p.o.sb + h * p.o.sh;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int r = r0 + ty * 4 + j;
    if (r >= p.Sq) continue;
    float l = row_l[ty * 4 + j], m = row_m[ty * 4 + j];
    float inv = l > 0.f ? 1.f / l : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int d = tx + 32 * i;
      if (d < p.D) store_out(const_cast<void*>(p.o.ptr), p.o_dtype, obase + r * p.o.ss + d * p.o.sd, acc[j][i] * inv);
    }
    if (p.lse && tx == 0) p.lse[((int64_t)b * p.H + h) * p.Sq + r] = l > 0.f ? m + log2f(l) : -CUDART_INF_F;
  }
}

// ------------------------------------------------------------------------ Dterm = scale * rowsum(dO * O)
__global__ void dterm_kernel(AttnParams p) {
  const int warps_per_block = blockDim.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int64_t rows = (int64_t)p.B * p.H * p.Sq;
  if (row >= rows) return;
  int s = (int)(row % p.Sq);
  int64_t bh = row / p.Sq;
  int h = (int)(bh % p.H), b = (int)(bh / p.H);
  const int64_t ob = b * p.o.sb + h * p.o.sh + s * p.o.ss;
  const int64_t gb = b * p.d_o.sb + h * p.d_o.sh + s * p.d_o.ss;
  float acc = 0.f;
  for (int d = lane; d < p.D; d += 32)
    acc = fmaf(load_elem(p.o.ptr, p.o_dtype, ob + d * p.o.sd), load_elem(p.d_o.ptr, p.do_dtype, gb + d * p.d_o.sd), acc);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) p.dterm[row] = acc * p.scale;
}

// ------------------------------------------------------------------------------------------- dQ
__global__ void __launch_bounds__(NT) bwd_dq_simt_kernel(AttnParams p) {
  extern __shared__ float smem[];
  const int Dp = (p.D + 31) & ~31, ld = Dp + 1;
  float* Qs = smem;
  float* dOs = Qs + TR * ld;
  float* Ks = dOs + TR * ld;
  float* Vs = Ks + TC * ld;
  float* Ss = Vs + TC * ld;            // dS tile [TR][TC+1]
  float* row_L = Ss + TR * (TC + 1);
  float* row_D = row_L + TR;

  const int b = blockIdx.z, h = blockIdx.y, r0 = blockIdx.x * TR;
  const int hk = h / (p.H / p.Hkv);
  const int ty = threadIdx.x >> 5, tx = threadIdx.x & 31;
  const int nbq = p.qq.block_rows > 0 ? (p.Sq + p.qq.block_rows - 1) / p.qq.block_rows : 1;
  const int nbk = p.qk.block_rows > 0 ? (p.Skv + p.qk.block_rows - 1) / p.qk.block_rows : 1;
  const int nbv = p.qv.block_rows > 0 ? (p.Skv + p.qv.block_rows - 1) / p.qv.block_rows : 1;
  QuantView none = {nullptr, 1.f, 0, 0};

  const int64_t sbq = ((int64_t)b * p.H + h) * nbq, sbk = ((int64_t)b * p.Hkv + hk) * nbk, sbv = ((int64_t)b * p.Hkv + hk) * nbv;
  load_tile(Qs, ld, p.q, p.in_dtype, p.qq, b, h, sbq, r0, TR, p.Sq, p.D, Dp);
  load_tile(dOs, ld, p.d_o, p.do_dtype, none, b, h, 0, r0, TR, p.Sq, p.D, Dp);
  if (threadIdx.x < TR) {
    int r = r0 + threadIdx.x;
    int64_t i = ((int64_t)b * p.H + h) * p.Sq + r;
    row_L[threadIdx.x] = r < p.Sq ? p.lse[i] : -CUDART_INF_F;
    row_D[threadIdx.x] = r < p.Sq ? p.dterm[i] : 0.f;
  }
  float acc[4][8];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[j][i] = 0.f;

  __shared__ int rlo[TR], rhi[TR];      // visible keys of each row
  if (threadIdx.x < TR) row_key_range(p.causal, p.window, p.Sq, p.Skv, p.cu_q, p.cu_k, p.nseq, r0 + threadIdx.x, rlo[threadIdx.x], rhi[threadIdx.x]);
  int klo, khi;
  block_key_range(p.causal, p.window, p.Sq, p.Skv, p.cu_q, p.cu_k, p.nseq, r0, min(r0 + TR, p.Sq), klo, khi);
  klo = (klo / TC) * TC;
  for (int c0 = klo; c0 < khi; c0 += TC) {
    __syncthreads();
    load_tile(Ks, ld, p.k, p.in_dtype, p.qk, b, hk, sbk, c0, TC, p.Skv, p.D, Dp);
    load_tile(Vs, ld, p.v, p.in_dtype, p.qv, b, hk, sbv, c0, TC, p.Skv, p.D, Dp);
    __syncthreads();
    float s[4], dp[4];
    tile_abt(Qs, Ks, ld, Dp, s);
    tile_abt(dOs, Vs, ld, Dp, dp);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int r = ty * 4 + j;
      float z = logit(p, b, h, r0 + r, c0 + tx, s[j], c0 + tx >= rlo[r] && c0 + tx < rhi[r]);
      float L = row_L[r];
      float pv = (L == -CUDART_INF_F) ? 0.f : exp2f(z - L);
      Ss[r * (TC + 1) + tx] = pv * (dp[j] * p.scale - row_D[r]);
    }
    __syncthreads();
    tile_acc<false>(Ss, TC + 1, Ks, ld, Dp, acc);
  }
  const int64_t base = (((int64_t)b * p.H + h) * p.Sq) * p.D;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int r = r0 + ty * 4 + j;
    if (r >= p.Sq) continue;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int d = tx + 32 * i;
      if (d < p.D) p.dq[base + (int64_t)r * p.D + d] = acc[j][i];
    }
  }
}

// ------------------------------------------------------------------------------------------- dK, dV
// One CTA per (32-key tile, kv head, batch); loops over the query heads sharing this kv head (GQA) and over
// query tiles, so dK/dV need no atomics.
__global__ void __launch_bounds__(NT) bwd_dkv_simt_kernel(AttnParams p) {
  extern __shared__ float smem[];
  const int Dp = (p.D + 31) & ~31, ld = Dp + 1;
  float* Ks = smem;
  float* Vs = Ks + TR * ld;
  float* Qs = Vs + TR * ld;
  float* dOs = Qs + TC * ld;
  float* Ps = dOs + TC * ld;            // P^T tile stored [key][query+1]
  float* dSs = Ps + TR * (TC + 1);      // dS^T tile
  float* row_L = dSs + TR * (TC + 1);   // per query of the inner tile
  float* row_D = row_L + TC;

  const int b = blockIdx.z, hk = blockIdx.y, c0 = blockIdx.x * TR;
  const int group = p.H / p.Hkv;
  const int ty = threadIdx.x >> 5, tx = threadIdx.x & 31;
  const int nbq = p.qq.block_rows > 0 ? (p.Sq + p.qq.block_rows - 1) / p.qq.block_rows : 1;
  const int nbk = p.qk.block_rows > 0 ? (p.Skv + p.qk.block_rows - 1) / p.qk.block_rows : 1;
  const int nbv = p.qv.block_rows > 0 ? (p.Skv + p.qv.block_rows - 1) / p.qv.block_rows : 1;
  QuantView none = {nullptr, 1.f, 0, 0};

  load_tile(Ks, ld, p.k, p.in_dtype, p.qk, b, hk, ((int64_t)b * p.Hkv + hk) * nbk, c0, TR, p.Skv, p.D, Dp);
  load_tile(Vs, ld, p.v, p.in_dtype, p.qv, b, hk, ((int64_t)b * p.Hkv + hk) * nbv, c0, TR, p.Skv, p.D, Dp);
  float dk[4][8], dv[4][8];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int i = 0; i < 8; ++i) { dk[j][i] = 0.f; dv[j][i] = 0.f; }

  __shared__ int kqlo[TR], kqhi[TR];    // query rows that see each key
  if (threadIdx.x < TR) key_query_range(p.causal, p.window, p.Sq, p.Skv, p.cu_q, p.cu_k, p.nseq, c0 + threadIdx.x, kqlo[threadIdx.x], kqhi[threadIdx.x]);
  int qlo, qhi;
  block_query_range(p.causal, p.window, p.Sq, p.Skv, p.cu_q, p.cu_k, p.nseq, c0, min(c0 + TR, p.Skv), qlo, qhi);
  qlo = (qlo / TC) * TC;
  for (int g = 0; g < group; ++g) {
    const int h = hk * group + g;
    for (int r0 = qlo; r0 < qhi; r0 += TC) {
      __syncthreads();
      load_tile(Qs, ld, p.q, p.in_dtype, p.qq, b, h, ((int64_t)b * p.H + h) * nbq, r0, TC, p.Sq, p.D, Dp);
      load_tile(dOs, ld, p.d_o, p.do_dtype, none, b, h, 0, r0, TC, p.Sq, p.D, Dp);
      if (threadIdx.x < TC) {
        int r = r0 + threadIdx.x;
        int64_t i = ((int64_t)b * p.H + h) * p.Sq + r;
        row_L[threadIdx.x] = r < p.Sq ? p.lse[i] : -CUDART_INF_F;
        row_D[threadIdx.x] = r < p.Sq ? p.dterm[i] : 0.f;
      }
      __syncthreads();
      // S^T[key][query]: thread rows = keys ty*4.., column = query tx
      float s[4], dp[4];
      tile_abt(Ks, Qs, ld, Dp, s);
      tile_abt(Vs, dOs, ld, Dp, dp);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        int kc = ty * 4 + j;
        float z = logit(p, b, h, r0 + tx, c0 + kc, s[j], r0 + tx >= kqlo[kc] && r0 + tx < kqhi[kc]);
        float L = row_L[tx];
        float pv = (L == -CUDART_INF_F) ? 0.f : exp2f(z - L);
        Ps[kc * (TC + 1) + tx] = pv;
        dSs[kc * (TC + 1) + tx] = pv * (dp[j] * p.scale - row_D[tx]);
      }
      __syncthreads();
      tile_acc<false>(Ps, TC + 1, dOs, ld, Dp, dv);
      tile_acc<false>(dSs, TC + 1, Qs, ld, Dp, dk);
    }
  }
  const int64_t base = (((int64_t)b * p.Hkv + hk) * p.Skv) * p.D;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int c = c0 + ty * 4 + j;
    if (c >= p.Skv) continue;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int d = tx + 32 * i;
      if (d < p.D) {
        p.dk[base + (int64_t)c * p.D + d] = dk[j][i];
        p.dv[base + (int64_t)c * p.D + d] = dv[j][i];
      }
    }
  }
}

template <typename K>
cudaError_t set_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

}  // namespace

cudaError_t launch_fwd_simt(const AttnParams& p, cudaStream_t st) {
  if (p.D > MAXD || p.D <= 0) return cudaErrorInvalidValue;
  const int Dp = (p.D + 31) & ~31, ld = Dp + 1;
  size_t smem = sizeof(float) * ((size_t)(TR + 2 * TC) * ld + TR * (TC + 1) + 3 * TR);
  cudaError_t e = set_smem(fwd_simt_kernel, smem);
  if (e != cudaSuccess) return e;
  dim3 grid((p.Sq + TR - 1) / TR, p.H, p.B);
  if (grid.x == 0 || grid.y == 0 || grid.z == 0) return cudaSuccess;
  fwd_simt_kernel<<<grid, NT, smem, st>>>(p);
  ++g_launch_count;
  g_last_kernel = "fwd_simt";
  return cudaGetLastError();
}

// Vector path: O fp32 and dO 16-bit, unit inner strides, D % 4 == 0, 16-byte aligned rows.  Each lane owns 4 adjacent
// elements per 128-wide slice (float4 of O, 8 bytes of dO); HBM-bound: 6 bytes per element in, 4 bytes per row out.
// A warp owns R consecutive rows and issues the loads of all of them before the first use: 24 R bytes in flight per lane
// (one row per warp left the memory system at 0.53 of the HBM rate, profiles/r01f_*; 4 rows per warp: 0.84).
template <bool BF16, int R>
__global__ void __launch_bounds__(256) dterm_vec_kernel(AttnParams p) {
  // grid = (row blocks of one (b, h), B * H): no 64-bit divisions on the way to the row pointers
  const int s0 = (int)((blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * R);
  const int lane = threadIdx.x & 31;
  if (s0 >= p.Sq) return;
  const int h = (int)(blockIdx.y % (unsigned)p.H), b = (int)(blockIdx.y / (unsigned)p.H);
  const int64_t row0 = ((int64_t)b * p.H + h) * p.Sq + s0;
  const int64_t rows = row0 - s0 + p.Sq;                     // end of this (b, h)
  const float* o[R];
  const uint16_t* g[R];
#pragma unroll
  for (int i = 0; i < R; ++i) {
    const int s = min(s0 + i, p.Sq - 1);                     // rows past the end repeat the last one (not written)
    o[i] = reinterpret_cast<const float*>(p.o.ptr) + b * p.o.sb + h * p.o.sh + s * p.o.ss;
    g[i] = reinterpret_cast<const uint16_t*>(p.d_o.ptr) + b * p.d_o.sb + h * p.d_o.sh + s * p.d_o.ss;
  }
  float acc[R];
#pragma unroll
  for (int i = 0; i < R; ++i) acc[i] = 0.f;
  for (int d = lane * 4; d < p.D; d += 128) {
    float4 ov[R];
    uint2 gv[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
      ov[i] = *reinterpret_cast<const float4*>(o[i] + d);
      gv[i] = *reinterpret_cast<const uint2*>(g[i] + d);
    }
#pragma unroll
    for (int i = 0; i < R; ++i) {
      float g0, g1, g2, g3;
      if (BF16) {
        g0 = __uint_as_float(gv[i].x << 16); g1 = __uint_as_float(gv[i].x & 0xffff0000u);
        g2 = __uint_as_float(gv[i].y << 16); g3 = __uint_as_float(gv[i].y & 0xffff0000u);
      } else {
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&gv[i].x));
        const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&gv[i].y));
        g0 = a.x; g1 = a.y; g2 = c.x; g3 = c.y;
      }
      acc[i] = fmaf(ov[i].x, g0, acc[i]); acc[i] = fmaf(ov[i].y, g1, acc[i]);
      acc[i] = fmaf(ov[i].z, g2, acc[i]); acc[i] = fmaf(ov[i].w, g3, acc[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < R; ++i) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], off);
  }
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < R; ++i)
      if (row0 + i < rows) p.dterm[row0 + i] = acc[i] * p.scale;
  }
}

cudaError_t launch_dterm(const AttnParams& p, cudaStream_t st) {
  int64_t rows = (int64_t)p.B * p.H * p.Sq;
  if (rows == 0) return cudaSuccess;
  const bool vec = p.o_dtype == kF32 && (p.do_dtype == kBF16 || p.do_dtype == kF16) && p.o.sd == 1 && p.d_o.sd == 1 &&
                   (p.D % 4) == 0 && !(reinterpret_cast<uintptr_t>(p.o.ptr) & 15) && !(reinterpret_cast<uintptr_t>(p.d_o.ptr) & 7) &&
                   !((p.o.ss | p.o.sh | p.o.sb) & 3) && !((p.d_o.ss | p.d_o.sh | p.d_o.sb) & 3);
  if (vec && (int64_t)p.B * p.H <= 65535) {
    // rows per warp (8 warps per block): 4 -- FLUX shape, 85 MB in: 24.0 us with 1 row per warp, 20.0 with 2,
    // 15.5 us = 5.5 TB/s = 0.84 of the measured copy rate with 4 (profiles/r02be_launches_dterm*.csv)
    constexpr int R = 4;
    const dim3 nb((unsigned)((p.Sq + 8 * R - 1) / (8 * R)), (unsigned)(p.B * p.H));
    if (p.do_dtype == kBF16) dterm_vec_kernel<true, R><<<nb, 256, 0, st>>>(p);
    else dterm_vec_kernel<false, R><<<nb, 256, 0, st>>>(p);
  } else {
    dterm_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(p);
  }
  ++g_launch_count;
  return cudaGetLastError();
}

cudaError_t launch_bwd_dkv_only(const AttnParams& p, cudaStream_t st) {
  if (p.D > MAXD || p.D <= 0 || !p.dk || !p.dv || !p.dterm) return cudaErrorInvalidValue;
  if (p.Skv <= 0 || p.B <= 0) return cudaSuccess;
  const int Dp = (p.D + 31) & ~31, ld = Dp + 1;
  size_t smem_kv = sizeof(float) * ((size_t)(2 * TR + 2 * TC) * ld + 2 * TR * (TC + 1) + 2 * TC);
  cudaError_t e = set_smem(bwd_dkv_simt_kernel, smem_kv);
  if (e != cudaSuccess) return e;
  dim3 grid((p.Skv + TR - 1) / TR, p.Hkv, p.B);
  bwd_dkv_simt_kernel<<<grid, NT, smem_kv, st>>>(p);
  ++g_launch_count;
  g_last_kernel = "bwd_simt";
  return cudaGetLastError();
}

cudaError_t launch_bwd_simt(const AttnParams& p, cudaStream_t st) {
  if (p.D > MAXD || p.D <= 0) return cudaErrorInvalidValue;
  cudaError_t e = launch_dterm(p, st);
  if (e != cudaSuccess) return e;
  const int Dp = (p.D + 31) & ~31, ld = Dp + 1;
  size_t smem_q = sizeof(float) * ((size_t)(2 * TR + 2 * TC) * ld + TR * (TC + 1) + 2 * TR);
  size_t smem_kv = sizeof(float) * ((size_t)(2 * TR + 2 * TC) * ld + 2 * TR * (TC + 1) + 2 * TC);
  if ((e = set_smem(bwd_dq_simt_kernel, smem_q)) != cudaSuccess) return e;
  if ((e = set_smem(bwd_dkv_simt_kernel, smem_kv)) != cudaSuccess) return e;
  if (p.Sq > 0 && p.B > 0 && p.dq) {
    dim3 grid((p.Sq + TR - 1) / TR, p.H, p.B);
    bwd_dq_simt_kernel<<<grid, NT, smem_q, st>>>(p);
    ++g_launch_count;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  if (p.Skv > 0 && p.B > 0 && p.dk && p.dv) {
    dim3 grid((p.Skv + TR - 1) / TR, p.Hkv, p.B);
    bwd_dkv_simt_kernel<<<grid, NT, smem_kv, st>>>(p);
    ++g_launch_count;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  g_last_kernel = "bwd_simt";
  return cudaSuccess;
}

}  // namespace mfa
