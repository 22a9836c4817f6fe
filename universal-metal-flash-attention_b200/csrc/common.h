// common.h -- shared host/device definitions for libMFAFFI.so (B200 / sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mfa {

// Element types, numbered like mfa_precision_t (include/mfa_ffi.h).
enum DType : int { kF16 = 0, kBF16 = 1, kF32 = 2, kI8 = 3, kI4 = 4 };

inline __host__ __device__ int dtype_bytes(int dt) { return dt == kF32 ? 4 : (dt == kI8 || dt == kI4) ? 1 : 2; }

enum MaskKind : int { kMaskNone = 0, kMaskBool = 1, kMaskAdditive = 2 };
enum MaskScalar : int { kMaskU8 = 0, kMaskF16 = 1, kMaskBF16 = 2, kMaskF32 = 3 };

// A [B, H, S, D] operand view: element (b,h,s,d) lives at ptr + b*sb + h*sh + s*ss + d*sd (element units).
// Contiguous BHSD has sd = 1, ss = D, sh = S*D, sb = H*S*D; transpose_x (reference: [D,S] per head) has
// ss = 1, sd = S.
struct TensorView {
  const void* ptr;
  int64_t sb, sh, ss, sd;
};

// Per-tensor / per-block symmetric quantisation metadata for an int8/int4 operand.
// block_rows tokens share one scale (0 = one scale for the whole tensor); scales laid out [B*H*ceil(S/block_rows)]
// when block_rows > 0.  value = (code - zero_point) * scale.
struct QuantView {
  const float* scales;   // device pointer, or nullptr -> use `scale`
  float scale;
  int zero_point;
  int block_rows;
};

struct AttnParams {
  TensorView q, k, v;       // inputs, in_dtype
  TensorView o;             // output (forward) or saved O (backward), o_dtype
  float* lse;               // [B,H,Sq] fp32, log2 units (L = log2e * logsumexp); may be null in forward
  int64_t lse_sh;           // forward, tensor-core path: elements between L rows of consecutive (b,h) (0 = Sq)
  int accumulate;           // forward, tensor-core path: merge the result into the (O, L) already in o / lse
  // backward only
  TensorView d_o;           // dO, do_dtype
  float* dq;                // fp32, contiguous BHSD
  float* dk;
  float* dv;
  float* dterm;             // [B,H,Sq] fp32: scale * rowsum(dO*O)
  int B, H, Hkv, Sq, Skv, D;
  float scale;
  int causal;               // key j visible to query i iff j <= i
  int window;               // <0: none; else hidden iff i > j + window
  // external mask, broadcast via zero strides
  const void* mask;
  int mask_kind, mask_scalar;
  int64_t mask_sb, mask_sh, mask_sq, mask_sk;
  // tensor-core forward: device scratch for the per-query-block lists of KV tiles the mask leaves visible (tile skipping);
  // null = every tile in the causal / window range is visited.  Size: fwd_tc_mask_scratch_bytes(p).
  int* mask_tile_scratch;
  int in_dtype, o_dtype, do_dtype;
  QuantView qq, qk, qv;     // used when in_dtype is kI8 / kI4
  // packed variable-length sequences (B == 1): device int32 offsets [nseq + 1] of the segments along the query / key axis;
  // null = dense.  See row_key_range.
  const int* cu_q;
  const int* cu_k;
  int nseq;
};

// Visible key range [lo, hi) for query rows [r0, r1) under causal/window rules (used for tile skipping).
__host__ __device__ inline void visible_key_range(int causal, int window, int Skv, int r0, int r1, int& lo, int& hi) {
  lo = 0; hi = Skv;
  if (causal) { int h = r1; if (h < hi) hi = h; }            // cols <= r1-1
  if (window >= 0) { int l = r0 - window; if (l > lo) lo = l; } // cols >= r0 - window
  if (hi < lo) hi = lo;
}

// Visible query range [lo, hi) for key columns [c0, c1).
__host__ __device__ inline void visible_query_range(int causal, int window, int Sq, int c0, int c1, int& lo, int& hi) {
  lo = 0; hi = Sq;
  if (causal) { if (c0 > lo) lo = c0; }                        // rows >= c0
  if (window >= 0) { long h = (long)c1 - 1 + window + 1; if (h < hi) hi = (int)h; } // rows <= c1-1+window
  if (hi < lo) hi = lo;
}

// ---- packed variable-length sequences.  Segment s holds query rows [cu_q[s], cu_q[s+1]) and keys [cu_k[s], cu_k[s+1]); a row
// sees the keys of its own segment only, and causal / window apply to the offsets inside the segment (top-left aligned):
// row i' = r - cu_q[s] hides key j' = c - cu_k[s] iff (causal && j' > i') || (window >= 0 && i' > j' + window).
// Offsets come from device memory the host has not checked: every bound derived from them is clamped to [0, total], so a
// malformed array gives wrong numbers but no access out of bounds.  cu == null is the dense problem (one segment, no clamps
// needed).  Per-row lower and upper key bounds never decrease with the row (and per-key query bounds with the key), so the
// range of a block of rows / keys is the lower bound of its first and the upper bound of its last.

__host__ __device__ inline int seg_offset(const int* cu, int s, int total) {
  const int v = cu[s];
  return v < 0 ? 0 : v > total ? total : v;
}

// s in [0, nseq) with cu[s] <= t < cu[s+1] (binary search; 0 / nseq - 1 past either end)
__host__ __device__ inline int segment_of(const int* cu, int nseq, int t) {
  int lo = 0, hi = nseq - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (cu[mid] <= t) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Visible keys [lo, hi) of query row r.
__host__ __device__ inline void row_key_range(int causal, int window, int Sq, int Skv, const int* cu_q, const int* cu_k, int nseq,
                                              int r, int& lo, int& hi) {
  if (!cu_q) {
    lo = window >= 0 ? max(0, r - window) : 0;
    hi = (causal ? min(Skv - 1, r) : Skv - 1) + 1;
    return;
  }
  const int s = segment_of(cu_q, nseq, r);
  const int i = r - seg_offset(cu_q, s, Sq);
  const int kb = seg_offset(cu_k, s, Skv);
  int ke = seg_offset(cu_k, s + 1, Skv);
  if (ke < kb) ke = kb;
  lo = kb; hi = ke;
  if (causal && i < ke - kb) hi = kb + (i < 0 ? 0 : i + 1);             // j' <= i'
  if (window >= 0 && i > window) lo = i - window < ke - kb ? kb + (i - window) : ke;   // j' >= i' - window
  if (hi < lo) hi = lo;
}

// Query rows [lo, hi) that see key c.  Dense: not clipped at Sq (rows past Sq carry L = +inf, P = 0).
__host__ __device__ inline void key_query_range(int causal, int window, int Sq, int Skv, const int* cu_q, const int* cu_k, int nseq,
                                                int c, int& lo, int& hi) {
  if (!cu_k) {
    lo = causal ? c : 0;
    hi = (window >= 0 ? min(c + window, 1 << 30) : (1 << 30)) + 1;
    return;
  }
  const int s = segment_of(cu_k, nseq, c);
  int j = c - seg_offset(cu_k, s, Skv);
  const int qb = seg_offset(cu_q, s, Sq);
  int qe = seg_offset(cu_q, s + 1, Sq);
  if (qe < qb) qe = qb;
  if (j < 0) j = 0;
  lo = qb; hi = qe;
  if (causal) lo = j < qe - qb ? qb + j : qe;                            // i' >= j'
  if (window >= 0 && (long long)j + window + 1 < qe - qb) hi = qb + j + window + 1;   // i' <= j' + window
  if (hi < lo) hi = lo;
}

// Visible keys [lo, hi) of query rows [r0, r1), r1 > r0.
__host__ __device__ inline void block_key_range(int causal, int window, int Sq, int Skv, const int* cu_q, const int* cu_k, int nseq,
                                                int r0, int r1, int& lo, int& hi) {
  if (!cu_q) { visible_key_range(causal, window, Skv, r0, r1, lo, hi); return; }
  int l2, h2;
  row_key_range(causal, window, Sq, Skv, cu_q, cu_k, nseq, r0, lo, h2);
  row_key_range(causal, window, Sq, Skv, cu_q, cu_k, nseq, r1 - 1, l2, hi);
  if (hi < lo) hi = lo;
}

// Query rows [lo, hi) that see any of the keys [c0, c1), c1 > c0.
__host__ __device__ inline void block_query_range(int causal, int window, int Sq, int Skv, const int* cu_q, const int* cu_k, int nseq,
                                                  int c0, int c1, int& lo, int& hi) {
  if (!cu_k) { visible_query_range(causal, window, Sq, c0, c1, lo, hi); return; }
  int l2, h2;
  key_query_range(causal, window, Sq, Skv, cu_q, cu_k, nseq, c0, lo, h2);
  key_query_range(causal, window, Sq, Skv, cu_q, cu_k, nseq, c1 - 1, l2, hi);
  if (hi < lo) hi = lo;
}

// ---- decode over a K/V cache.  Sequence b holds L_b valid keys, the last Sq of them the new tokens: query row s sits at position
// p = L_b - Sq + s and sees key j < L_b iff (!causal || j <= p) && (window < 0 || p - j <= window) (bottom-right alignment).
// L_b comes from device memory the host has not checked: kvc_len clamps it to [0, capacity].  Per-row bounds never decrease with
// s, so the range of a block of rows is the lower bound of its first and the upper bound of its last.

__host__ __device__ inline int kvc_len(const int* lens, int b, int cap) {
  const int v = lens[b];
  return v < 0 ? 0 : v > cap ? cap : v;
}

// Visible keys [lo, hi) of query row s (lo == hi: none).
__host__ __device__ inline void kvc_row_key_range(int causal, int window, int L, int Sq, int s, int& lo, int& hi) {
  const int p = L - Sq + s;
  lo = window >= 0 ? max(0, p - window) : 0;
  hi = causal ? min(L, p + 1) : L;
  if (hi < lo) hi = lo;
}

// Visible keys [lo, hi) of query rows [s0, s1), s1 > s0.
__host__ __device__ inline void kvc_block_key_range(int causal, int window, int L, int Sq, int s0, int s1, int& lo, int& hi) {
  int l2, h2;
  kvc_row_key_range(causal, window, L, Sq, s0, lo, h2);
  kvc_row_key_range(causal, window, L, Sq, s1 - 1, l2, hi);
  if (hi < lo) hi = lo;
}

// A per-sequence number of new tokens (cu_q: sequence b owns query rows [cu[b], cu[b+1]) of total_q, at most max_sq of them).
// Offsets come from memory the host may not have checked: they are clamped to [0, total_q] (seg_offset), and sq_b to
// [0, max_sq], so the rows of a segment past max_sq are rows that see no key.
__host__ __device__ inline int kvc_seq_len(const int* cu, int b, int total, int max_sq) {
  const int n = seg_offset(cu, b + 1, total) - seg_offset(cu, b, total);
  return n < 0 ? 0 : n > max_sq ? max_sq : n;
}

// Packed item slots: with T query tokens per work item, sequence b's items start at slot cu[b] / T + b.  That is strictly
// increasing in b and leaves each sequence at least ceil(sq_b / T) slots, total_q / T + num_seqs slots in all.
__host__ __device__ inline int kvc_first_slot(const int* cu, int b, int total, int T) { return seg_offset(cu, b, total) / T + b; }

// The sequence whose slots hold `slot` (binary search; 0 before the first).
__host__ __device__ inline int kvc_slot_owner(const int* cu, int nseq, int total, int T, int slot) {
  int lo = 0, hi = nseq - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (kvc_first_slot(cu, mid, total, T) <= slot) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Key tiles [t0, t1) of split k when the ntiles 128-key tiles of the capacity are shared by nsplit splits.
__host__ __device__ inline void kvc_split_tiles(int ntiles, int nsplit, int k, int& t0, int& t1) {
  const int per = (ntiles + nsplit - 1) / nsplit;
  t0 = min(k * per, ntiles);
  t1 = min(t0 + per, ntiles);
}

// Log2-domain merge of attention partials over disjoint key sets (SURVEY 8e): with m = max_k L_k and w_k = 2^(L_k - m),
//   L = m + log2(sum_k w_k),  O = sum_k O_k w_k / sum_k w_k.
// A partial without keys (L_k = -inf) weighs 0.  With one partial, w = 1 and L = m exactly.
__device__ __forceinline__ float lse_merge_weight(float lk, float m) { return lk == -__int_as_float(0x7f800000) ? 0.f : exp2f(lk - m); }
__device__ __forceinline__ float lse_merge_total(float m, float wsum) { return m + log2f(wsum); }

// Rotary embedding of one pair: (x0, x1) -> (x0 c - x1 s, x0 s + x1 c) in fp32, each product pair fused the same way in every
// kernel that rotates (rope_kernel, kvcache_append_kernel), so their outputs agree bit for bit.
__device__ __forceinline__ void rope_pair(float x0, float x1, float c, float s, float& y0, float& y1) {
  y0 = __fmaf_rn(x0, c, -__fmul_rn(x1, s));
  y1 = __fmaf_rn(x0, s, __fmul_rn(x1, c));
}

// Writing new tokens' K / V into a K/V cache (mfa_kvcache_append), K and optionally Q rotated on the way.  Token s of sequence b
// goes to cache row p = L_b - sq_b + s (the decode rule above) and reads rotary table row p.
struct KvAppendParams {
  TensorView q, q_out;       // [B, H, Sq, D] views (with cu_q [1, H, total_q, D]); q.ptr == null: Q is not rotated
  TensorView k_new, v_new;   // [B, Hkv, Sq, D] views (with cu_q [1, Hkv, total_q, D])
  TensorView k, v;           // caches as in KvCacheParams
  const int* seqlens;        // [B] device
  const int* block_table;    // [B, cap / page_size] device, or null (contiguous cache)
  const int* cu_q;           // [B + 1] device query offsets, or null: Sq new tokens per sequence
  const float* cos_t;        // fp32 [rotary_rows, rotary_dim / 2] (one angle per pair), or null: no rotation
  const float* sin_t;
  int rotary_rows, rotary_dim, interleaved;   // interleaved: pairs (2i, 2i+1); else half-split pairs (i, i + rotary_dim / 2)
  int B, H, Hkv, Sq, D, cap, page_size, num_pages;   // with cu_q, Sq is max_seqlen_q
  int total_q;               // token rows in all (B * Sq without cu_q)
  int dtype;                 // kBF16 or kF16
};
cudaError_t launch_kvcache_append(const KvAppendParams& p, cudaStream_t st);

// Attention of new tokens per sequence against that sequence's K/V cache (mfa_attention_forward_kvcache and, with cu_q,
// mfa_attention_forward_kvcache_varlen).
struct KvCacheParams {
  TensorView q, o;           // [B, H, Sq, D] views (o in o_dtype); with cu_q [1, H, total_q, D]
  TensorView k, v;           // contiguous cache: [B, Hkv, cap, D] views; paged: base of the [num_pages, page_size, Hkv, D] pools
  float* lse;                // [B, H, Sq] or null; with cu_q [H, total_q]
  const int* seqlens;        // [B] device
  const int* block_table;    // [B, cap / page_size] device, or null (contiguous cache)
  const int* cu_q;           // [B + 1] device query offsets, or null: Sq new tokens per sequence
  int B, H, Hkv, Sq, D, cap, page_size, num_pages;   // with cu_q, Sq is the largest number of new tokens (max_seqlen_q)
  int total_q;               // query rows in all (B * Sq without cu_q)
  float scale;
  int causal, window, in_dtype, o_dtype;
};
// How a call is cut into work items: G query heads per KV head share a tile as rows g * sqb + s (rows = G * sqb live rows), a
// work item holds two such tiles of consecutive tokens, and the keys of the capacity are shared by nsplit splits.  The items of
// one KV head and split sit in query-item slots: nqi per sequence, or with cu_q whichever is fewer of that and the packed
// slots (kvc_first_slot, slots != 0).  Chosen from the shape and the SM count only, never from the lengths.
struct KvCachePlan {
  int G, sqb, rows, nqi, nsplit;
  int slots;                 // packed slots, or 0: nqi slots per sequence
  long long items;
  size_t o_bytes, l_bytes;   // scratch: partial O (fp32 [items][2][rows][D]) and L ([items][2][rows])
};
KvCachePlan kvcache_plan(const KvCacheParams& p, int sm_count);
cudaError_t launch_fwd_kvcache(const KvCacheParams& p, const KvCachePlan& plan, void* scratch, cudaStream_t st);

// ---- kernel launchers (each returns cudaGetLastError()) ----
cudaError_t launch_fwd_simt(const AttnParams& p, cudaStream_t st);
cudaError_t launch_bwd_simt(const AttnParams& p, cudaStream_t st);          // dterm + dQ + dK/dV
cudaError_t launch_dterm(const AttnParams& p, cudaStream_t st);
cudaError_t launch_bwd_dkv_only(const AttnParams& p, cudaStream_t st);      // dK/dV from a caller-supplied dterm

// tcgen05 forward (bf16/fp16, D in {64,128}); returns cudaErrorNotSupported when the problem is not eligible.
bool fwd_tc_eligible(const AttnParams& p);
size_t fwd_tc_mask_scratch_bytes(const AttnParams& p);     // 0 when there is no external mask
size_t bwd_tc_mask_scratch_bytes(const AttnParams& p);     // same for the backward's two list sets
void mask_tile_dims(const AttnParams& p, int& nqb, int& nkt, int& MB, int& MH);
cudaError_t launch_mask_flags(const AttnParams& p, uint8_t* flags, cudaStream_t st);
cudaError_t launch_fwd_tc(const AttnParams& p, cudaStream_t st);

// tcgen05 backward (bf16/fp16, D in {64,128}); needs p.dterm filled by launch_dterm first.
bool bwd_tc_eligible(const AttnParams& p);
cudaError_t launch_bwd_tc(const AttnParams& p, cudaStream_t st);

// fp32 operands on the tensor pipe as fp16 (hi, lo) pairs (attn_fwd_split.cu): head_dim 128
bool fwd_split_eligible(const AttnParams& p);
size_t fwd_split_scratch_bytes(const AttnParams& p);
cudaError_t launch_fwd_split(const AttnParams& p, void* scratch, cudaStream_t st);

// int8 tensor-core forward (attn_fwd_tcq.cu): int8 / int4 codes, symmetric, D = 128, per-tensor or 64-multiple block scales.
bool fwd_tcq_eligible(const AttnParams& p);
size_t fwd_tcq_scratch_bytes(const AttnParams& p);
cudaError_t launch_fwd_tcq(const AttnParams& p, void* scratch, cudaStream_t st);
cudaError_t launch_codes_to_bf16(const void* codes, int bits, void* dst, uint64_t n, cudaStream_t st);
int fwd_tcq_pv_mode();                      // P V of the quantised tensor-core forward: 0 = e4m3 (default), 1 = bf16
void fwd_tcq_set_pv_mode(int bf16);

// quantiser & friends
cudaError_t launch_quantize(const void* src, int src_dtype, void* codes, float* scales, uint64_t rows, uint64_t cols,
                            uint32_t block_rows, uint32_t block_cols, int bits, float scale_floor, cudaStream_t st);
cudaError_t launch_dequantize(const void* codes, const float* scales, float* out, uint64_t rows, uint64_t cols,
                              uint32_t block_rows, uint32_t block_cols, int bits, cudaStream_t st);
// tensor-core backward of quantised operands: dequantised codes / the upstream gradient as bf16
cudaError_t launch_dequantize_bf16(const void* codes, int bits, const QuantView& q, void* out, uint64_t heads,
                                   uint64_t rows_per_head, uint32_t D, cudaStream_t st);
cudaError_t launch_to_bf16(const void* src, int src_dtype, void* out, uint64_t n, cudaStream_t st);
cudaError_t launch_merge_partials(float* o_acc, float* l_acc, const float* o_part, const float* l_part,
                                  uint64_t rows, uint32_t D, cudaStream_t st);
cudaError_t launch_hadamard(float* data, uint32_t block_size, uint32_t num_blocks, cudaStream_t st);
cudaError_t launch_rope(const void* src, void* dst, const float* cos_t, const float* sin_t, int64_t sB, int64_t sH,
                        int64_t sS, int64_t table_batch_stride, bool negate_sin, uint32_t B, uint32_t H, uint32_t S,
                        uint32_t D, int dtype, cudaStream_t st);
cudaError_t launch_convert_from_f32(const float* src, void* dst, int dst_dtype, uint64_t n, cudaStream_t st);

// Count of kernel launches performed by this library (bench.py's gpu_launches claim).
extern unsigned long long g_launch_count;
extern const char* g_last_kernel;

}  // namespace mfa
