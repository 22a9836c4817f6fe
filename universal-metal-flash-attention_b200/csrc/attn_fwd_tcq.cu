// attn_fwd_tcq.cu -- front end of the quantised attention forward on the sm_100a tensor pipe (SageAttention2-style):
//     S_int = Q_i8 K_i8^T            tcgen05.mma kind::i8 (int32 accumulator in TMEM, 2x the bf16 MMA rate)
//     S     = S_int * qs[row block] * ks[key block]          (fp32, in the softmax warps)
//   P V in e4m3 (default; BASELINE.json config 3 "int8 Q K^T and fp8 P V"):
//     P'    = 2^6 exp2(S c - m) -> e4m3 in TMEM,  O += P' V_e4m3      (kind::f8f6f4, 2x the bf16 MMA rate, half the V bytes);
//             V_e4m3 = e4m3(code * vs[key block] / vh) with one scale vh per (b, head), applied to O in the epilogue
//   P V in bf16 (mfa_set_quantized_pv_precision(ctx, MFA_PRECISION_BF16)):
//     P     = exp2(S c - m)  -> bf16 in TMEM,  O += (P * vs[key block]) V_codes      (kind::f16, V codes exact in bf16)
// Replaces the reference's quantised forward (metal-flash-attention/Sources/FlashAttention/Attention/
// QuantizedAttention.swift:71-91,358-463 -- attention on dequantised int8 operands with fp32 statistics) for symmetric
// int8 codes (zero_point 0) with per-tensor or per-block scales (block = a multiple of 64 tokens of one (b, h); the
// SageAttention2 contract SURVEY Q5 settles on), head_dim 128.  The fused kernel is the int8 operand mode of
// attn_fwd_tc.cu (same pipeline, masking and P hand-off; packed int4 Q / K are unpacked in shared
// memory by its converter warp); this file holds the HBM-bound pre-passes over V (codes -> e4m3 or bf16), eligibility and
// parameter set-up.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <math_constants.h>
#include <cstring>

#include "common.h"
#include "fwd_tc.h"
#include "sm100_ptx.cuh"
#include "tc_host.h"

namespace mfa {

namespace {

using namespace ptx;

constexpr float kLog2e = 1.4426950408889634f;

// ---- HBM-bound pre-passes over V (Q and K go to the MMA as they are: int8 codes through TMA, packed int4 through TMA + the
// in-kernel converter warp) -----------------------------------------------------------------------------------------------
// 16 codes of V as ints: int8 bytes, or packed int4 (byte j = codes 2j | 2j+1 << 4, each stored + 8: GEMMQuantization.swift:501-516)
template <int BITS>
__device__ __forceinline__ void load_codes16(const uint8_t* __restrict__ src, uint64_t i, int* q) {
  if (BITS == 8) {
    const int4 v = reinterpret_cast<const int4*>(src)[i];
    const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 16; ++k) q[k] = (int)(int8_t)((w[k >> 2] >> (8 * (k & 3))) & 0xff);
  } else {
    const uint2 v = reinterpret_cast<const uint2*>(src)[i];
    const uint32_t w[2] = {v.x, v.y};
#pragma unroll
    for (int k = 0; k < 16; ++k) q[k] = (int)((w[k >> 3] >> (4 * (k & 7))) & 0xf) - 8;
  }
}

// V codes -> bf16 (exact: |code| <= 128 needs 8 significant bits); 16 codes per thread per step.
template <int BITS>
__global__ void codes_to_bf16_kernel(const uint8_t* __restrict__ src, __nv_bfloat16* __restrict__ dst, uint64_t n16) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n16; i += (uint64_t)gridDim.x * blockDim.x) {
    int q[16];
    load_codes16<BITS>(src, i, q);
    uint32_t out[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) out[k] = pack_bf16((float)q[2 * k], (float)q[2 * k + 1]);
    reinterpret_cast<uint4*>(dst)[2 * i] = make_uint4(out[0], out[1], out[2], out[3]);
    reinterpret_cast<uint4*>(dst)[2 * i + 1] = make_uint4(out[4], out[5], out[6], out[7]);
  }
}

// ---- e4m3 V for the fp8 P V path.  One fp32 scale per (b, head): vh = max over the head's blocks of (block scale) * qmax / 448,
// so every dequantised value code * vs[block] maps into e4m3's range (|x / vh| <= 448); e4m3 is a floating format, so one scale
// per head loses no relative precision against per-block scales.  Pass 1 reads the scale array only.
__global__ void head_vscale_kernel(const float* __restrict__ scales, float one_scale, int nb_per_head, int heads, float qmax,
                                   float* __restrict__ vh) {
  const int hd = blockIdx.x * blockDim.x + threadIdx.x;
  if (hd >= heads) return;
  float mx = 0.f;
  if (scales && nb_per_head > 0) for (int i = 0; i < nb_per_head; ++i) mx = fmaxf(mx, scales[(size_t)hd * nb_per_head + i]);
  else mx = scales ? scales[0] : one_scale;
  const float v = mx * qmax * (1.f / 448.f);
  vh[hd] = v > 0.f ? v : 1.f;
}

// V codes -> e4m3(code * vs[block] / vh[head]); 16 codes per thread per step, a (b, head) spans rows_per_head * D elements
template <int BITS>
__global__ void codes_to_e4m3_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, const float* __restrict__ scales,
                                     float one_scale, const float* __restrict__ vh, int block_rows, int nb_per_head,
                                     uint64_t rows_per_head, uint32_t D, uint64_t n16) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n16; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t e = i * 16;
    const uint64_t row = e / D;
    const uint64_t hd = row / rows_per_head;
    float sc = one_scale;
    if (scales) sc = nb_per_head > 0 ? scales[hd * nb_per_head + (row - hd * rows_per_head) / block_rows] : scales[0];
    const float r = sc / vh[hd];
    int q[16];
    load_codes16<BITS>(src, i, q);
    uint32_t out[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      out[k] = pack_e4m3((float)q[4 * k] * r, (float)q[4 * k + 1] * r) | (pack_e4m3((float)q[4 * k + 2] * r, (float)q[4 * k + 3] * r) << 16);
    reinterpret_cast<uint4*>(dst)[i] = make_uint4(out[0], out[1], out[2], out[3]);
  }
}

unsigned __float_as_uint_host(float f) { unsigned u; memcpy(&u, &f, 4); return u; }

unsigned grid_for(uint64_t n, int threads) {
  uint64_t g = (n + threads - 1) / threads;
  const uint64_t cap = 148ull * 16;
  return (unsigned)(g < cap ? (g ? g : 1) : cap);
}

int g_tcq_pv = 0;        // 0 = e4m3 P V (default), 1 = bf16 P V

bool scales_ok(const QuantView& q, bool need64) {
  if (q.zero_point != 0) return false;
  if (!q.scales || q.block_rows == 0) return q.block_rows == 0;     // one scale: by value, or scales[0] on the device
  if (q.block_rows < 0) return false;
  return !need64 || (q.block_rows % 64) == 0;
}

}  // namespace

cudaError_t launch_codes_to_bf16(const void* codes, int bits, void* dst, uint64_t n, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  if (n % 16) return cudaErrorInvalidValue;
  if (bits == 8)
    codes_to_bf16_kernel<8><<<grid_for(n / 16, 256), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(codes), reinterpret_cast<__nv_bfloat16*>(dst), n / 16);
  else
    codes_to_bf16_kernel<4><<<grid_for(n / 16, 256), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(codes), reinterpret_cast<__nv_bfloat16*>(dst), n / 16);
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace mfa

namespace mfa {
// P V precision of the quantised tensor-core forward: e4m3 (default) or bf16
int fwd_tcq_pv_mode() { return g_tcq_pv; }
void fwd_tcq_set_pv_mode(int bf16) { g_tcq_pv = bf16 ? 1 : 0; }

// Eligibility of the int8 tensor-core forward: int8 or int4 codes, symmetric, head_dim 128, contiguous operands, per-tensor
// scales or per-block scales with K / V blocks that are multiples of 64 tokens, no external mask.
bool fwd_tcq_eligible(const AttnParams& p) {
  if (getenv("MFA_DISABLE_TC")) return false;
  if (p.in_dtype != kI8 && p.in_dtype != kI4) return false;
  if (p.D != 128 || !fwd_tc_mask_ok(p)) return false;
  if (!(p.scale > 0.f) || p.Sq <= 0 || p.Skv <= 0 || p.B <= 0 || p.H <= 0 || p.Hkv <= 0 || p.H % p.Hkv) return false;
  if (p.B > 65535 || p.H > 65535) return false;
  // V: the bf16 P V path folds its block scales into the exponent per 64-key half; the e4m3 path takes any block size
  if (!scales_ok(p.qq, false) || !scales_ok(p.qk, true) || !scales_ok(p.qv, fwd_tcq_pv_mode() == 1)) return false;
  const TensorView* vs[3] = {&p.q, &p.k, &p.v};
  const int64_t S[3] = {p.Sq, p.Skv, p.Skv}, Hn[3] = {p.H, p.Hkv, p.Hkv};
  for (int i = 0; i < 3; ++i) {      // contiguous BHSD (the pre-passes work on flat arrays)
    if (vs[i]->sd != 1 || vs[i]->ss != p.D || vs[i]->sh != S[i] * p.D || vs[i]->sb != Hn[i] * S[i] * p.D) return false;
    if (reinterpret_cast<uintptr_t>(vs[i]->ptr) & 15) return false;
  }
  if (p.o.sd != 1) return false;
  const int oes = dtype_bytes(p.o_dtype);
  if ((reinterpret_cast<uintptr_t>(p.o.ptr) & 15) || ((p.o.ss * oes) & 15) || ((p.o.sh * oes) & 15) || ((p.o.sb * oes) & 15))
    return false;
  return tc::encode_fn() != nullptr;
}

// scratch: Skv*B*Hkv*D*2 bytes (V as bf16; the e4m3 path uses half of it) + B*Hkv head scales
size_t fwd_tcq_scratch_bytes(const AttnParams& p) {
  const size_t nkv = (size_t)p.B * p.Hkv * p.Skv * p.D;
  return nkv * 2 + (size_t)p.B * p.Hkv * 4 + 2048;
}

cudaError_t launch_fwd_tcq(const AttnParams& p, void* scratch, cudaStream_t st) {
  const size_t nkv = (size_t)p.B * p.Hkv * p.Skv * p.D;
  uint8_t* sc = reinterpret_cast<uint8_t*>(scratch);
  void* v16 = sc;
  const void *qc = p.q.ptr, *kc = p.k.ptr, *vc = p.v.ptr;
  const bool i4 = p.in_dtype == kI4;
  const int bits = i4 ? 4 : 8;
  cudaError_t e;
  const bool f8 = fwd_tcq_pv_mode() == 0;
  float* vh = nullptr;                      // e4m3 path: one scale per (b, head), behind V in the scratch
  if (nkv % 16) return cudaErrorInvalidValue;
  if (f8) {
    const size_t off = (nkv * 2 + 1023) & ~(size_t)255;
    vh = reinterpret_cast<float*>(sc + off);
    const int heads = p.B * p.Hkv;
    const bool blocks = p.qv.scales && p.qv.block_rows > 0;
    const int nb = blocks ? (p.Skv + p.qv.block_rows - 1) / p.qv.block_rows : 0;
    const float qmax = i4 ? 8.f : 128.f;
    head_vscale_kernel<<<(heads + 127) / 128, 128, 0, st>>>(p.qv.scales, p.qv.scale, nb, heads, qmax, vh);
    if (i4)
      codes_to_e4m3_kernel<4><<<grid_for(nkv / 16, 256), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(vc), reinterpret_cast<uint8_t*>(v16),
                                                                      p.qv.scales, p.qv.scale, vh, blocks ? p.qv.block_rows : 1, nb,
                                                                      (uint64_t)p.Skv, (uint32_t)p.D, nkv / 16);
    else
      codes_to_e4m3_kernel<8><<<grid_for(nkv / 16, 256), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(vc), reinterpret_cast<uint8_t*>(v16),
                                                                      p.qv.scales, p.qv.scale, vh, blocks ? p.qv.block_rows : 1, nb,
                                                                      (uint64_t)p.Skv, (uint32_t)p.D, nkv / 16);
    g_launch_count += 2;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  } else if ((e = launch_codes_to_bf16(vc, bits, v16, nkv, st)) != cudaSuccess) {
    return e;
  }

  FwdTcParams prm = {};
  TensorView tq = p.q, tk = p.k, tv = p.v;
  tq.ptr = qc; tk.ptr = kc; tv.ptr = v16;
  if (i4) {     // packed rows of D / 2 bytes, unpacked by the kernel's converter warp
    if (!tc::make_map_raw(&prm.tq, qc, p.B, p.H, p.Sq, p.D / 2) || !tc::make_map_raw(&prm.tk, kc, p.B, p.Hkv, p.Skv, p.D / 2))
      return cudaErrorInvalidValue;
  } else if (!tc::make_map(&prm.tq, tq, kI8, p.B, p.H, p.Sq, p.D) || !tc::make_map(&prm.tk, tk, kI8, p.B, p.Hkv, p.Skv, p.D)) {
    return cudaErrorInvalidValue;
  }
  if (!tc::make_map(&prm.tv, tv, f8 ? kI8 : kBF16, p.B, p.Hkv, p.Skv, p.D)) return cudaErrorInvalidValue;
  prm.o = const_cast<void*>(p.o.ptr);
  prm.o_sb = p.o.sb; prm.o_sh = p.o.sh; prm.o_ss = p.o.ss;
  prm.lse = p.lse; prm.o_dtype = p.o_dtype;
  prm.lse_sh = p.lse_sh > 0 ? p.lse_sh : p.Sq;
  prm.H = p.H; prm.Hkv = p.Hkv; prm.Sq = p.Sq; prm.Skv = p.Skv;
  prm.c = p.scale * kLog2e;
  prm.causal = p.causal; prm.window = p.window;
  fwd_tc_set_mask(prm, p);
  if ((e = fwd_tc_build_mask_tiles(prm, p, st)) != cudaSuccess) return e;
  fwd_tc_set_out_map(prm, p);
  auto setq = [](const QuantView& q, int S, const float*& arr, float& one, int& br, int& nb, int& stride) {
    arr = q.scales; one = q.scale;
    const bool blocks = q.scales && q.block_rows > 0;
    br = blocks ? q.block_rows : 1 << 30;
    nb = blocks ? (S + q.block_rows - 1) / q.block_rows : 1;
    stride = blocks ? nb : 0;
  };
  setq(p.qq, p.Sq, prm.qs, prm.qs1, prm.qbr, prm.nbq, prm.sq_);
  setq(p.qk, p.Skv, prm.ks, prm.ks1, prm.kbr, prm.nbk, prm.sk_);
  setq(p.qv, p.Skv, prm.vs, prm.vs1, prm.vbr, prm.nbv, prm.sv_);
  {   // |S_int| <= 128 * 128 * 128 = 2^21 (int8) or 8 * 8 * 128 = 2^13 (int4): the widest shift whose +-2^(22-k) window holds it
    const int k = i4 ? 8 : 1;          // int4: q in [-8, 7] times UNSIGNED k nibbles in [0, 15], |S_mma| <= 8 * 15 * 128 < 2^14
    prm.s_mul = 1 << k;
    prm.s_bias = 1.5f * (float)(1u << (23 - k));
    prm.s_add = __float_as_uint_host(prm.s_bias);
  }
  if (f8) { prm.vs = vh; prm.vs1 = 1.f; }        // e4m3 V: the kernel reads vs[b * Hkv + head] in its epilogue
  e = launch_fwd_tc_kernel(prm, p.D, i4 ? (f8 ? kFwdI4F8 : kFwdI4) : (f8 ? kFwdI8F8 : kFwdI8), st, p.B);
  if (e != cudaSuccess) return e;
  ++g_launch_count;
  g_last_kernel = f8 ? (p.in_dtype == kI4 ? "fwd_tcq_int4_pvf8_d128" : "fwd_tcq_int8_pvf8_d128")
                     : (p.in_dtype == kI4 ? "fwd_tcq_int4_d128" : "fwd_tcq_int8_d128");
  return cudaGetLastError();
}

}  // namespace mfa
