// fwd_tc.h -- parameter block and launcher of the fused tcgen05 attention forward (attn_fwd_tc.cu), shared with the
// quantised front end (attn_fwd_tcq.cu), which runs the same kernel with the int8 Q K^T operand mode.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include "common.h"

namespace mfa {

// I8: int8 Q K^T + bf16 P V; I8F8: int8 Q K^T + e4m3 P V; Split: fp32 operands as scaled fp16 (hi, lo) pairs, three MMAs per product
// I4 / I4F8: as I8 / I8F8 with Q and K delivered as packed int4 and unpacked in shared memory (tq / tk map the packed bytes)
// WideF16 / WideBF16: head_dim 256 as two 128-column halves -- a CTA computes S over all 256 dims (two MMA groups) and ONE half of O
// (the TMEM budget is 2 tiles x (S 128 + O 128) columns), so the grid doubles and Q K^T runs twice
enum FwdMode : int { kFwdF16 = 0, kFwdBF16 = 1, kFwdI8 = 2, kFwdI8F8 = 3, kFwdSplit = 4, kFwdI4 = 5, kFwdI4F8 = 6,
                     kFwdWideF16 = 7, kFwdWideBF16 = 8 };

struct FwdTcParams {
  CUtensorMap tq, tk, tv;
  CUtensorMap tq2, tk2, tv2;   // kFwdSplit: the lo halves (tq / tk / tv map the hi halves)
  CUtensorMap to;          // O in its output type, box = 128 bytes (32 floats / 64 halves) x 128 rows (valid when o_tma != 0)
  int o_tma;               // epilogue stages O in shared memory and writes it with TMA bulk stores
  void* o;
  long long o_sb, o_sh, o_ss;
  float* lse;
  long long lse_sh;        // elements between the L rows of consecutive (b, h) pairs (Sq unless the output is a row window)
  int accumulate;          // merge this launch's partial (O, L) with what lse / o already hold (fp32 O, lse required)
  int o_dtype;
  int H, Hkv, Sq, Skv;
  int dv;                  // true head dim when it is smaller than the kernel's tile width (0 = the full width): direct stores stop there
  int nbatch;              // set by launch_fwd_tc_kernel (work items = query blocks x H x nbatch)
  float c;                 // softmax_scale * log2(e)
  int causal, window;
  int flush_steps;         // kFwdSplit: O leaves TMEM for an fp32 scratch tile every flush_steps KV steps (0 = never)
  float* flush_buf;        // [work items][2 tiles][D / 4][128 rows][4] floats
  // kFwdI8 only: symmetric scales of the int8 codes (value = code * scale)
  const float* qs; const float* ks; const float* vs;   // per-block scale arrays (device) or nullptr
  float qs1, ks1, vs1;                                  // per-tensor scales when the array is null
  int qbr, kbr, vbr;                                    // tokens per block (multiple of 64 for K / V)
  int nbq, nbk, nbv;                                    // blocks per (b, h)
  int sq_, sk_, sv_;                                    // scale-array stride per (b, h): nb, or 0 for a single device scale
  // int32 score -> float without a conversion: bits(s * s_mul + s_add) = s_bias + s  (s_mul = 2^k, s_bias = 1.5 * 2^(23-k))
  int s_mul; unsigned s_add; float s_bias;
  // external mask (kernels instantiated with MASKED): bool bytes (non-zero = attend) or additive values, element strides
  // over [B, H, Sq, Skv] with broadcast dims = 0 and mask_sk == 1
  const void* mask;
  int mask_kind, mask_scalar;
  long long mask_sb, mask_sh, mask_sq;
  // dense 1- / 2-byte masks: tiles staged in shared memory by TMA (tm over [MB, MH, Sq, Skv], box 128 bytes x 128 rows); only
  // read by the MASKED instantiations of the modes that have the room (not int4 / split / wide)
  CUtensorMap tm;
  int mask_tma;
  // tile skipping under an external mask: per (mask batch, mask head, query block) a compacted list of the KV tiles that
  // hold at least one visible element (built by mask_tiles_kernel right before the launch), or null
  const int* mtiles;       // [lists][m_nkt]
  const int* mcounts;      // [lists]
  int m_nkt;
  const int* cu_q;         // packed variable-length sequences (AttnParams::cu_q / cu_k / nseq), or null
  const int* cu_k;
  int nseq;
  // decode over a K/V cache (common.h, kvc_*) when kv_len is set; read by the unmasked 16-bit instantiations only.  A work item is
  // (query item, split, KV head, sequence), query items fastest; its tiles hold the G query heads of one KV head as rows g * kv_sqb + s (tq is the 5-D
  // (D, Sq, G, Hkv, B) map), and it leaves a normalised partial: O through `to` at (column, 0, tile, item) and L in
  // lse[(item * 2 + tile) * kv_rows + row].
  const int* kv_len;       // [B] valid keys per sequence
  const int* kv_pages;     // [B][kv_npb] page table, or null (contiguous cache: tk / tv map [B, Hkv, cap, D])
  int kv_cap, kv_page, kv_npages, kv_npb, kv_box;   // capacity, page size, pages in the pool, pages per sequence, rows per K / V box
  int kv_g, kv_sqb, kv_rows, kv_nqi, kv_nsplit;     // see KvCachePlan
  int kv_qbytes;           // bytes TMA writes into one Q tile
  // per-sequence new tokens: sequence b owns query rows [kv_cu_q[b], kv_cu_q[b+1]) of kv_total, at most Sq of them, and tq is
  // the (D, kv_total, G, Hkv, 1) map.  Null: Sq rows per sequence.  kv_slots != 0: packed slots (common.h, kvc_first_slot);
  // a work item is then (slot, split, KV head), slots fastest.
  const int* kv_cu_q;
  int kv_total, kv_slots;
};

bool fwd_tc_mask_ok(const AttnParams& p);
void fwd_tc_set_mask(FwdTcParams& prm, const AttnParams& p);
cudaError_t fwd_tc_build_mask_tiles(FwdTcParams& prm, const AttnParams& p, cudaStream_t st);
void fwd_tc_set_out_map(FwdTcParams& prm, const AttnParams& p);

// grid = (ceil(Sq / 256), H, B).  mode kFwdI8 needs D == 128 (Q / K tiles are int8, V tiles bf16).
cudaError_t launch_fwd_tc_kernel(const FwdTcParams& prm, int D, int mode, cudaStream_t st, int B);

}  // namespace mfa
