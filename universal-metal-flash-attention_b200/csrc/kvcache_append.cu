// kvcache_append.cu -- writes the new tokens' K / V into a contiguous or paged K/V cache in one launch, rotating K (and
// optionally Q) on the way (mfa_kvcache_append).  HBM-bound: every element is read once and written once with 16-byte vector
// accesses along D; no scratch, no allocation, so the launch can sit in a CUDA graph in front of the attention call.
//
// One CTA per new token.  Thread 0 finds the token's sequence (one binary search over cu_q), its cache row p = L_b - sq_b + s
// and, in a paged cache, the page; the CTA then walks the token's Q, K and V head rows in units of 16 bytes.  A unit of a rotated
// row holds both members of each of its pairs: four interleaved pairs (2i, 2i+1) of one 8-element chunk, or, half-split, the
// 8-element chunks at i and i + rotary_dim / 2, so no thread needs another's data.  Columns from rotary_dim to D are copied.
// The append is kept out of the attention kernel on purpose: several work items of one sequence (key splits, query items) read
// the new keys, so writing them from inside the attention would race with those reads.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.h"

namespace mfa {
namespace {

constexpr int kThreads = 256;

template <typename T> __device__ __forceinline__ float to_f(T x);
template <> __device__ __forceinline__ float to_f<__half>(__half x) { return __half2float(x); }
template <> __device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 x) { return __bfloat162float(x); }
template <typename T> __device__ __forceinline__ T from_f(float x);
template <> __device__ __forceinline__ __half from_f<__half>(float x) { return __float2half_rn(x); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }

// 8 elements <-> fp32 through one 16-byte register vector
template <typename T> __device__ __forceinline__ void unpack8(const uint4& raw, float x[8]) {
  const T* e = reinterpret_cast<const T*>(&raw);
#pragma unroll
  for (int i = 0; i < 8; ++i) x[i] = to_f<T>(e[i]);
}
template <typename T> __device__ __forceinline__ uint4 pack8(const float x[8]) {
  uint4 raw;
  T* e = reinterpret_cast<T*>(&raw);
#pragma unroll
  for (int i = 0; i < 8; ++i) e[i] = from_f<T>(x[i]);
  return raw;
}

__device__ __forceinline__ uint4 ld16(const void* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void st16(void* p, const uint4& v) { *reinterpret_cast<uint4*>(p) = v; }
__device__ __forceinline__ float4 ld_table(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// Unit u of one rotated head row: src / dst point at element 0 of the row, cs / sn at the token's table row.  nhalf = the number of
// half-split pair units (rotary_dim / 16; 0 for interleaved or no rotation), rd = rotary_dim.
template <typename T>
__device__ __forceinline__ void rotate_unit(const T* src, T* dst, const float* cs, const float* sn, int u, int nhalf, int rd) {
  if (u < nhalf) {                                    // half-split: pairs (i, i + rd / 2) for i in [8u, 8u + 8)
    const int c0 = 8 * u, c1 = c0 + rd / 2;
    const uint4 ra = ld16(src + c0), rb = ld16(src + c1);
    const float4 ca = ld_table(cs + c0), cb = ld_table(cs + c0 + 4), sa = ld_table(sn + c0), sb = ld_table(sn + c0 + 4);
    const float c[8] = {ca.x, ca.y, ca.z, ca.w, cb.x, cb.y, cb.z, cb.w}, s[8] = {sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z, sb.w};
    float a[8], b[8];
    unpack8<T>(ra, a);
    unpack8<T>(rb, b);
#pragma unroll
    for (int i = 0; i < 8; ++i) rope_pair(a[i], b[i], c[i], s[i], a[i], b[i]);
    st16(dst + c0, pack8<T>(a));
    st16(dst + c1, pack8<T>(b));
    return;
  }
  const int col = 8 * (u + nhalf);
  const uint4 raw = ld16(src + col);
  if (col >= rd) { st16(dst + col, raw); return; }    // past rotary_dim: copied unrotated
  const float4 c = ld_table(cs + col / 2), s = ld_table(sn + col / 2);   // interleaved: pairs (2i, 2i + 1), i in [col/2, col/2 + 4)
  float x[8];
  unpack8<T>(raw, x);
  rope_pair(x[0], x[1], c.x, s.x, x[0], x[1]);
  rope_pair(x[2], x[3], c.y, s.y, x[2], x[3]);
  rope_pair(x[4], x[5], c.z, s.z, x[4], x[5]);
  rope_pair(x[6], x[7], c.w, s.w, x[6], x[7]);
  st16(dst + col, pack8<T>(x));
}

template <typename T>
__global__ void __launch_bounds__(kThreads) kvcache_append_kernel(const KvAppendParams p) {
  __shared__ int sh_b, sh_s, sh_pos;
  __shared__ long long sh_row;               // paged: element offset of the cache row in the pools; contiguous: unused
  const int t = blockIdx.x;
  if (threadIdx.x == 0) {
    int b, s, sq;
    if (p.cu_q) {
      b = segment_of(p.cu_q, p.B, t);
      s = t - seg_offset(p.cu_q, b, p.total_q);
      sq = kvc_seq_len(p.cu_q, b, p.total_q, p.Sq);
    } else {
      b = t / p.Sq;
      s = t - b * p.Sq;
      sq = p.Sq;
    }
    const int L = kvc_len(p.seqlens, b, p.cap);
    const int pos = L - sq + s;              // < L <= cap
    long long row = 0;
    if (p.block_table && pos >= 0) {
      int page = p.block_table[(long long)b * (p.cap / p.page_size) + pos / p.page_size];
      page = page < 0 ? 0 : page >= p.num_pages ? p.num_pages - 1 : page;
      row = ((long long)page * p.page_size + pos % p.page_size) * p.Hkv * p.D;
    }
    sh_b = b; sh_s = (s >= 0 && s < sq) ? s : -1; sh_pos = pos; sh_row = row;
  }
  __syncthreads();
  const int s = sh_s;
  if (s < 0) return;                         // outside every segment, or past max_seqlen_q: nothing is written
  const int b = sh_b, pos = sh_pos;
  const long long tok = p.cu_q ? 0 : b;      // view batch index and row of the token in the q / k_new / v_new views
  const long long trow = p.cu_q ? t : s;
  const int D = p.D, D8 = D / 8, rd = p.cos_t ? p.rotary_dim : 0;
  const int nhalf = (rd && !p.interleaved) ? rd / 16 : 0;
  const int U = D8 - nhalf;                  // units of a rotated row
  int r = pos < 0 ? 0 : pos >= p.rotary_rows ? p.rotary_rows - 1 : pos;   // table row (Q rows use the clamped position)
  if (r < 0) r = 0;
  const float* cs = p.cos_t + (long long)r * (rd / 2);
  const float* sn = p.sin_t + (long long)r * (rd / 2);
  const int nq = p.q.ptr ? p.H * U : 0;
  const int nk = pos >= 0 ? p.Hkv * U : 0;   // K / V rows with p < 0 are not written
  const int nv = pos >= 0 ? p.Hkv * D8 : 0;
  const T* kn = reinterpret_cast<const T*>(p.k_new.ptr) + tok * p.k_new.sb + trow * p.k_new.ss;
  const T* vn = reinterpret_cast<const T*>(p.v_new.ptr) + tok * p.v_new.sb + trow * p.v_new.ss;
  T* kc = const_cast<T*>(reinterpret_cast<const T*>(p.k.ptr));
  T* vc = const_cast<T*>(reinterpret_cast<const T*>(p.v.ptr));
  long long k_sh = (long long)D, v_sh = (long long)D;
  if (p.block_table) {
    kc += sh_row; vc += sh_row;
  } else {
    kc += b * p.k.sb + (long long)pos * p.k.ss; vc += b * p.v.sb + (long long)pos * p.v.ss;
    k_sh = p.k.sh; v_sh = p.v.sh;
  }
  for (int i = threadIdx.x; i < nq + nk + nv; i += kThreads) {
    if (i < nq) {
      const int h = i / U;
      const T* src = reinterpret_cast<const T*>(p.q.ptr) + tok * p.q.sb + h * p.q.sh + trow * p.q.ss;
      T* dst = const_cast<T*>(reinterpret_cast<const T*>(p.q_out.ptr)) + tok * p.q_out.sb + h * p.q_out.sh + trow * p.q_out.ss;
      rotate_unit<T>(src, dst, cs, sn, i - h * U, nhalf, rd);
    } else if (i < nq + nk) {
      const int j = i - nq, h = j / U;
      rotate_unit<T>(kn + h * p.k_new.sh, kc + h * k_sh, cs, sn, j - h * U, nhalf, rd);
    } else {
      const int j = i - nq - nk, h = j / D8, col = 8 * (j - h * D8);
      st16(vc + h * v_sh + col, ld16(vn + h * p.v_new.sh + col));
    }
  }
}

}  // namespace

cudaError_t launch_kvcache_append(const KvAppendParams& p, cudaStream_t st) {
  const long long tokens = p.cu_q ? p.total_q : (long long)p.B * p.Sq;
  if (tokens <= 0) return cudaSuccess;
  if (p.dtype == kBF16) {
    kvcache_append_kernel<__nv_bfloat16><<<(unsigned)tokens, kThreads, 0, st>>>(p);
    g_last_kernel = "kvcache_append_bf16";
  } else if (p.dtype == kF16) {
    kvcache_append_kernel<__half><<<(unsigned)tokens, kThreads, 0, st>>>(p);
    g_last_kernel = "kvcache_append_fp16";
  } else {
    return cudaErrorInvalidValue;
  }
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace mfa
