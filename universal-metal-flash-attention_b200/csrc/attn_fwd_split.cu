// attn_fwd_split.cu -- fp32 operands on the sm_100a tensor pipe: front end of the kFwdSplit mode of attn_fwd_tc.cu.
//
// fp32 is the default precision of every adapter of the reference (strings default to fp32: Sources/MFABridge/
// MFABridge.swift:1438-1451; the Rust / Objective-C examples pass fp32), whose Metal kernels then run fp32 simdgroup
// matrix products (AttentionDescriptor+Precisions.swift:143-146).  tcgen05 has no fp32 MMA, so each operand is split
// into two fp16 tensors
//     x * 2^k = hi + lo,   hi = f16(x 2^k),  lo = f16(x 2^k - hi)          (22 significant bits; 2^k puts max|x| into [2^13, 2^14))
// and every product runs as three kind::f16 MMAs into the same fp32 TMEM accumulator,
//     S = Q_hi K_lo^T + Q_hi K_hi^T + Q_lo K_hi^T,      O += P_hi V_hi + P_lo V_hi + P_hi V_lo,
// P being split the same way by the softmax warps (P_hi / P_lo share the TMEM columns S has just left).  The dropped lo * lo
// terms are 2^-22 of a product, the fp16 products are exact and accumulate in fp32, the softmax itself is the fp32 code of
// the 16-bit kernel with MUFU exp2 only -- the result agrees with the fp64 oracle to ~5e-6 of max|O| (tests hold 1e-5; what
// limits it is the truncating accumulation of tcgen05.mma, see launch_fwd_split),
// at three times the MMA work of the bf16 kernel instead of the 9 TFLOP/s of the exact SIMT kernel it replaces at D = 128.
// The power-of-two scales are undone exactly: 2^-(kq + kk) rides in the softmax scale, 2^-kv in the epilogue's 1 / l.
//
// This file holds the HBM-bound pre-passes (abs-max per tensor, split into the (hi, lo) scratch tensors), eligibility and
// parameter set-up; the fused kernel is attn_fwd_tc.cu.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdlib>

#include "common.h"
#include "fwd_tc.h"
#include "tc_host.h"

namespace mfa {

namespace {

constexpr float kLog2e = 1.4426950408889634f;
constexpr int kSliceKeys = 768;       // keys per accumulator lifetime (a multiple of 128, see launch_fwd_split)

struct SplitView {
  const float* src;
  long long sb, sh, ss;        // element strides of the [B, H, S, D] source view (unit stride along D)
  int H, S, D4;                // D / 4
  int contiguous;              // packed BHSD: element index = linear index
  unsigned long long n4;       // B * H * S * D / 4
};

// float4 group i of the packed [B, H, S, D] order.  Contiguous sources (the common case) need no index arithmetic; strided
// ones pay three integer divisions per 16 bytes (still far cheaper than what the pass replaces).
__device__ __forceinline__ const float4* row_ptr(const SplitView& v, unsigned long long i, int& d4) {
  if (v.contiguous) { d4 = 0; return reinterpret_cast<const float4*>(v.src) + i; }
  d4 = (int)(i % v.D4);
  unsigned long long r = i / v.D4;
  const int s = (int)(r % v.S); r /= v.S;
  const int h = (int)(r % v.H);
  const long long b = (long long)(r / v.H);
  return reinterpret_cast<const float4*>(v.src + b * v.sb + (long long)h * v.sh + (long long)s * v.ss) + d4;
}

struct SplitViews { SplitView v[3]; };      // Q, K, V of one call: blockIdx.y picks the tensor, so each pre-pass is ONE launch

// exponent k of the power-of-two scale: max|x| 2^k in [2^13, 2^14), clamped so that 2^k and 2^-k stay normal floats
__device__ __forceinline__ int split_exponent(unsigned int amax_bits) {
  const float a = __uint_as_float(amax_bits);
  if (!(a > 0.f) || !isfinite(a)) return 0;
  int e;
  frexpf(a, &e);                       // a = m 2^e, m in [0.5, 1)
  return max(-100, min(100, 14 - e));
}

constexpr int kIlp = 4;                // independent 16-byte loads in flight per thread and pass

// max |x| per tensor: bit pattern of a non-negative float orders like the float, so one atomicMax per warp does it
__global__ void __launch_bounds__(256) split_absmax_kernel(const SplitViews vs, unsigned int* __restrict__ amax) {
  const SplitView& v = vs.v[blockIdx.y];
  float m = 0.f;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long i0 = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < v.n4; i0 += stride * kIlp) {
    float4 x[kIlp];
#pragma unroll
    for (int j = 0; j < kIlp; ++j) {
      const unsigned long long i = i0 + j * stride;
      int d4;
      x[j] = i < v.n4 ? __ldg(row_ptr(v, i, d4)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int j = 0; j < kIlp; ++j)
      m = fmaxf(fmaxf(m, fmaxf(fabsf(x[j].x), fabsf(x[j].y))), fmaxf(fabsf(x[j].z), fabsf(x[j].w)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(amax + blockIdx.y, __float_as_uint(m));
}

// hi / lo halves, packed [B, H, S, D] fp16 each (lo right behind hi); thread 0 leaves the inverse scale for the attention kernel
struct SplitOut { __half* hi[3]; };
__global__ void __launch_bounds__(256) split_f16_kernel(const SplitViews vs, const unsigned int* __restrict__ amax, const SplitOut out,
                                                        float* __restrict__ inv_scale) {
  const SplitView& v = vs.v[blockIdx.y];
  const int k = split_exponent(amax[blockIdx.y]);
  const float sc = ldexpf(1.f, k);
  if (blockIdx.x == 0 && threadIdx.x == 0) inv_scale[blockIdx.y] = ldexpf(1.f, -k);
  __half* hi = out.hi[blockIdx.y];
  __half* lo = hi + v.n4 * 4;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long i0 = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < v.n4; i0 += stride * kIlp) {
    float4 x[kIlp];
#pragma unroll
    for (int j = 0; j < kIlp; ++j) {
      const unsigned long long i = i0 + j * stride;
      int d4;
      if (i < v.n4) x[j] = __ldg(row_ptr(v, i, d4));
    }
#pragma unroll
    for (int j = 0; j < kIlp; ++j) {
      const unsigned long long i = i0 + j * stride;
      if (i >= v.n4) break;
      const float xs[4] = {x[j].x * sc, x[j].y * sc, x[j].z * sc, x[j].w * sc};
      __half h[4], l[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        h[c] = __float2half_rn(xs[c]);
        l[c] = __float2half_rn(xs[c] - __half2float(h[c]));
      }
      reinterpret_cast<uint2*>(hi)[i] = *reinterpret_cast<const uint2*>(h);
      reinterpret_cast<uint2*>(lo)[i] = *reinterpret_cast<const uint2*>(l);
    }
  }
}

bool src_ok(const TensorView& t, int64_t Hn, int64_t B) {
  if (t.sd != 1 || (reinterpret_cast<uintptr_t>(t.ptr) & 15)) return false;
  if (t.ss <= 0 || (t.ss & 3)) return false;
  if (Hn > 1 && (t.sh <= 0 || (t.sh & 3))) return false;
  if (B > 1 && (t.sb <= 0 || (t.sb & 3))) return false;
  return true;
}

size_t pad256(size_t x) { return (x + 255) & ~(size_t)255; }

unsigned split_grid(unsigned long long n4) {
  const unsigned long long g = (n4 + 255) / 256, cap = 148ull * 4;
  return (unsigned)(g < cap ? (g ? g : 1) : cap);
}

}  // namespace

// fp32 operands, head_dim 128, unit stride along D with 16-byte aligned rows; masks as for the 16-bit kernel
bool fwd_split_eligible(const AttnParams& p) {
  if (getenv("MFA_DISABLE_TC") || getenv("MFA_DISABLE_TC32")) return false;
  // head dims below 128 (multiples of 8) ride the same kernel: the (hi, lo) scratch tensors keep the true head dim, TMA zero-fills
  if (p.in_dtype != kF32 || p.D < 8 || p.D > 128 || (p.D & 7) || p.accumulate || !fwd_tc_mask_ok(p)) return false;
  if (!(p.scale > 0.f) || p.Sq <= 0 || p.Skv <= 0 || p.B <= 0 || p.H <= 0 || p.Hkv <= 0 || p.H % p.Hkv) return false;
  if (p.B > 65535 || p.H > 65535) return false;
  if (!src_ok(p.q, p.H, p.B) || !src_ok(p.k, p.Hkv, p.B) || !src_ok(p.v, p.Hkv, p.B)) return false;
  if (p.o.sd != 1) return false;
  const int oes = dtype_bytes(p.o_dtype);
  if ((reinterpret_cast<uintptr_t>(p.o.ptr) & 15) || ((p.o.ss * oes) & 15) || ((p.o.sh * oes) & 15) || ((p.o.sb * oes) & 15))
    return false;
  return tc::encode_fn() != nullptr;
}

// scratch: (hi, lo) fp16 copies of Q, K, V + three abs-max words + three inverse scales
size_t fwd_split_scratch_bytes(const AttnParams& p) {
  const size_t nq = (size_t)p.B * p.H * p.Sq * p.D, nkv = (size_t)p.B * p.Hkv * p.Skv * p.D;
  // + the flush tiles of the key slices (128 KB per 256-row work item)
  const size_t items = (size_t)((p.Sq + 255) / 256) * p.H * p.B;
  return pad256(nq * 4) + 2 * pad256(nkv * 4) + 512 + items * 2 * 128 * 128 * 4 + 256;
}

cudaError_t launch_fwd_split(const AttnParams& p, void* scratch, cudaStream_t st) {
  const size_t nq = (size_t)p.B * p.H * p.Sq * p.D, nkv = (size_t)p.B * p.Hkv * p.Skv * p.D;
  uint8_t* sc = reinterpret_cast<uint8_t*>(scratch);
  __half* qh = reinterpret_cast<__half*>(sc);
  __half* kh = reinterpret_cast<__half*>(sc + pad256(nq * 4));
  __half* vh = reinterpret_cast<__half*>(sc + pad256(nq * 4) + pad256(nkv * 4));
  unsigned int* amax = reinterpret_cast<unsigned int*>(sc + pad256(nq * 4) + 2 * pad256(nkv * 4));
  float* inv = reinterpret_cast<float*>(amax + 8);
  cudaError_t e = cudaMemsetAsync(amax, 0, 32, st);
  if (e != cudaSuccess) return e;
  const TensorView* src[3] = {&p.q, &p.k, &p.v};
  __half* dst[3] = {qh, kh, vh};
  const int Hn[3] = {p.H, p.Hkv, p.Hkv}, S[3] = {p.Sq, p.Skv, p.Skv};
  const size_t n[3] = {nq, nkv, nkv};
  SplitViews vs;
  SplitOut out;
  unsigned long long nmax = 0;
  for (int i = 0; i < 3; ++i) {
    const bool packed_src = src[i]->ss == p.D && src[i]->sh == (int64_t)S[i] * p.D && src[i]->sb == (int64_t)Hn[i] * S[i] * p.D;
    vs.v[i] = SplitView{reinterpret_cast<const float*>(src[i]->ptr), src[i]->sb, src[i]->sh, src[i]->ss, Hn[i], S[i], p.D / 4,
                        packed_src ? 1 : 0, n[i] / 4};
    out.hi[i] = dst[i];
    nmax = vs.v[i].n4 > nmax ? vs.v[i].n4 : nmax;
  }
  const dim3 grid(split_grid((nmax + kIlp - 1) / kIlp), 3, 1);
  split_absmax_kernel<<<grid, 256, 0, st>>>(vs, amax);
  split_f16_kernel<<<grid, 256, 0, st>>>(vs, amax, out, inv);
  g_launch_count += 2;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;

  FwdTcParams prm = {};
  auto packed = [&](const __half* ptr, int Hh, int Ss) {
    TensorView t;
    t.ptr = ptr; t.sd = 1; t.ss = p.D; t.sh = (int64_t)Ss * p.D; t.sb = (int64_t)Hh * Ss * p.D;
    return t;
  };
  if (!tc::make_map(&prm.tq, packed(qh, p.H, p.Sq), kF16, p.B, p.H, p.Sq, p.D) ||
      !tc::make_map(&prm.tq2, packed(qh + nq, p.H, p.Sq), kF16, p.B, p.H, p.Sq, p.D) ||
      !tc::make_map(&prm.tk, packed(kh, p.Hkv, p.Skv), kF16, p.B, p.Hkv, p.Skv, p.D) ||
      !tc::make_map(&prm.tk2, packed(kh + nkv, p.Hkv, p.Skv), kF16, p.B, p.Hkv, p.Skv, p.D) ||
      !tc::make_map(&prm.tv, packed(vh, p.Hkv, p.Skv), kF16, p.B, p.Hkv, p.Skv, p.D) ||
      !tc::make_map(&prm.tv2, packed(vh + nkv, p.Hkv, p.Skv), kF16, p.B, p.Hkv, p.Skv, p.D))
    return cudaErrorInvalidValue;
  prm.o = const_cast<void*>(p.o.ptr);
  prm.o_sb = p.o.sb; prm.o_sh = p.o.sh; prm.o_ss = p.o.ss;
  prm.lse = p.lse; prm.o_dtype = p.o_dtype;
  prm.lse_sh = p.lse_sh > 0 ? p.lse_sh : p.Sq;
  prm.accumulate = 0;
  prm.H = p.H; prm.Hkv = p.Hkv; prm.Sq = p.Sq; prm.Skv = p.Skv;
  prm.dv = p.D;
  prm.c = p.scale * kLog2e;
  prm.causal = p.causal; prm.window = p.window;
  prm.cu_q = p.cu_q; prm.cu_k = p.cu_k; prm.nseq = p.nseq;
  prm.qs = inv; prm.ks = inv + 1; prm.vs = inv + 2;          // inverse power-of-two scales, read by the softmax warps
  fwd_tc_set_out_map(prm, p);
  fwd_tc_set_mask(prm, p);
  // Long key ranges run as slices of kSliceKeys keys.  Why: tcgen05 adds every MMA into the TMEM accumulator with truncation, a
  // bias of ~2^-24 of the accumulator per MMA; O collects 24 MMAs per KV step, so one accumulator over N keys carries a relative
  // error of N * 4e-9 (zero-mean V) to N * 9e-9 (same-sign V, the accumulator grows monotonically): 1.7e-5 .. 4.2e-5 at 4608
  // keys -- beyond the 1e-5 this path promises.  Slices of 768 keys keep the worst case at ~7e-6 (2048: 1.7e-5, 1024: ~9e-6;
  // tests/test_gpu_fp32_tc.py).  The kernel hands O over to an fp32 scratch tile every kSliceKeys / 128 steps (one launch, no
  // re-read of Q, no extra prologues).
  if (!p.accumulate && p.Skv > kSliceKeys) {
    prm.flush_steps = kSliceKeys / 128;
    prm.flush_buf = reinterpret_cast<float*>(sc + pad256(nq * 4) + 2 * pad256(nkv * 4) + 512);
  }
  if ((e = fwd_tc_build_mask_tiles(prm, p, st)) != cudaSuccess) return e;
  e = launch_fwd_tc_kernel(prm, 128, kFwdSplit, st, p.B);
  if (e != cudaSuccess) return e;
  ++g_launch_count;
  g_last_kernel = prm.mask ? "fwd_tc_fp32split_d128_mask" : "fwd_tc_fp32split_d128";
  return cudaGetLastError();
}

}  // namespace mfa
