/*
 * mfa_ffi_ext.h -- symbols libMFAFFI.so exports beyond mfa_ffi.h.
 *
 * Part 1: the 13 symbols the reference's Swift bridge exports with @_cdecl but never declares in its
 *         header; its PyTorch adapter re-declares them by hand
 *         (examples/pytorch-custom-op-ffi/include/metal_sdpa_backend.h:312-534, src/mps_utils.mm:9-24).
 *         Prototypes here are the C spellings of the Swift signatures cited per function
 *         ("bridge:" = Sources/MFABridge/MFABridge.swift, "bridgeQ:" = Sources/MFABridge/MFABridge+Quantized.swift).
 * Part 2: additive B200 symbols (sliding window, CUDA streams, device quantiser, multi-GPU helpers).
 *         No existing prototype is changed.
 */
#ifndef MFA_FFI_EXT_H
#define MFA_FFI_EXT_H

#include "mfa_ffi.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ============================== Part 1: exported-but-undeclared reference symbols ============== */

/* bridge:1476 -- mfa_attention_forward with string precisions: "fp16"/"float16", "bf16"/"bfloat16",
 * "fp32"/"float32" (bridge:1438-1451; anything else = fp32). */
mfa_error_t mfa_attention_forward_str(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal,
    const char* input_precision, const char* intermediate_precision, const char* output_precision,
    bool transpose_q, bool transpose_k, bool transpose_v, bool transpose_o,
    const void* mask_ptr, size_t mask_size_bytes, const int64_t* mask_shape, const int64_t* mask_strides,
    uint32_t mask_ndim, mfa_mask_type_t mask_type, mfa_mask_scalar_t mask_scalar_type);

/* bridge:807 -- stores per-row scale arrays on the context; the reference never reads them back
 * (bridge:825-845).  Stored here too; consumed by the *_unified/_enhanced entry points when
 * granularity == 1 (row-wise) and the operands are pre-quantised. */
mfa_error_t mfa_set_scale_arrays(mfa_context_t context,
                                 const float* q_scales, uint32_t q_scales_count,
                                 const float* k_scales, uint32_t k_scales_count,
                                 const float* v_scales, uint32_t v_scales_count);

int32_t mfa_has_native_bfloat(void);         /* bridge:1550 -- 1 on B200 */
int32_t mfa_has_native_bfloat_msl32(void);   /* bridge:1576 -- 1 on B200 */

/* bridge:2671 / :2844 -- granularity 0 tensor, 1 row, 2 block, 3 hybrid (= block); *_block_size in tokens
 * (0 = 64).  Same operand rules as mfa_attention_forward_quantized. */
mfa_error_t mfa_attention_forward_quantized_unified(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    mfa_precision_t q_precision, mfa_precision_t k_precision, mfa_precision_t v_precision,
    mfa_precision_t output_precision, int32_t granularity,
    uint32_t q_block_size, uint32_t k_block_size, uint32_t v_block_size,
    bool enable_mixed_precision, bool force_symmetric_quantization,
    bool transpose_q, bool transpose_k, bool transpose_v, bool transpose_o);

mfa_error_t mfa_attention_forward_quantized_enhanced(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    mfa_precision_t q_precision, mfa_precision_t k_precision, mfa_precision_t v_precision,
    mfa_precision_t output_precision, int32_t granularity,
    uint32_t q_block_size, uint32_t k_block_size, uint32_t v_block_size,
    bool enable_mixed_precision, bool force_symmetric_quantization,
    bool transpose_q, bool transpose_k, bool transpose_v, bool transpose_o);

/* bridgeQ:12 -- "direct" runtime-quantising forward: q_precision = input element type (0 fp16, 1 bf16,
 * 2 fp32), k_precision = target (3 int8, 4 int4), v_precision = mode (0 tensor-wise, 2 block-wise(64));
 * the six scale/zero-point arguments are unused, as in the reference. */
mfa_error_t mfa_attention_forward_quantized_direct(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    int32_t q_precision, int32_t k_precision, int32_t v_precision, int32_t output_precision,
    bool transpose_q, bool transpose_k, bool transpose_v, bool transpose_o);

/* bridgeQ:178 */
mfa_error_t mfa_multihead_attention_quantized_direct(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    int32_t q_precision, int32_t k_precision, int32_t v_precision);

/* bridge:3078 -- forward that also returns L = log2(e) * logsumexp(scale * S), fp32 [B,H,Sq]. */
int32_t mfa_attention_forward_with_lse(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t lse,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t input_precision, int32_t intermediate_precision,
    bool transpose_q, bool transpose_k, bool transpose_v, bool transpose_o);

/* bridgeQ:227 -- quantise Q, K, V on the device (target_precision 3 int8 | 4 int4; quant_mode 0 per-tensor |
 * 2 per-block of 64 tokens), run attention, return O (fp32) and L.  mask: NULL or dense fp32 additive
 * [B,H,Sq,Skv].  input_precision uses the C enum (bridgeQ:273-278). */
int32_t mfa_quantized_forward_with_lse(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t lse,
    mfa_buffer_t mask,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t target_precision, int32_t quant_mode, int32_t input_precision);

/* bridgeQ:365 -- re-quantises Q, K, V deterministically, then dQ/dK/dV (fp32) on the dequantised operands;
 * grad_out is fp32; allocates its own D scratch (bridgeQ:475-478). */
int32_t mfa_quantized_backward(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    mfa_buffer_t grad_out, mfa_buffer_t lse, mfa_buffer_t grad_q, mfa_buffer_t grad_k, mfa_buffer_t grad_v,
    mfa_buffer_t mask,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t target_precision, int32_t quant_mode, int32_t input_precision);

/* bridge:3433 -- in-place fast Walsh-Hadamard transform over num_blocks blocks of block_size fp32 values
 * (power of two <= 1024), scaled by 1/sqrt(block_size).  No context argument, as in the reference. */
int32_t mfa_hadamard_rotate(mfa_buffer_t data, uint32_t block_size, uint32_t num_blocks);

/* bridge:2286 -- interleaved-pair RoPE encoded on a caller stream (command_buffer = cudaStream_t); buffers are
 * device pointers with byte offsets; strides in elements; cos/sin tables fp32, pair-duplicated [S, D] (or [B, S, D]):
 * element b * table_batch_stride + s * D + 2 * pair is read, table_batch_stride = 0 or S * D (bridge:282,305). */
int mfa_rope_rotate_encode_mtl(
    mfa_context_t context, void* command_buffer,
    void* src, int64_t src_offset, int64_t src_stride_b, int64_t src_stride_h, int64_t src_stride_s,
    void* dst, int64_t dst_offset,
    void* cos_table, int64_t cos_offset, void* sin_table, int64_t sin_offset, int64_t table_batch_stride,
    bool negate_sin, uint32_t batch_size, uint32_t num_heads, uint32_t seq_len, uint32_t head_dim,
    const char* precision);

/* ============================== Part 2: additive B200 symbols ================================== */

/* Forward with everything the engine supports.  lse may be NULL.  window_size < 0 = none; otherwise key j is
 * hidden from query i iff i > j + window_size (the reference kernel's rule, AttentionKernel+Softmax.swift:450,
 * which no mfa_* symbol reaches -- SURVEY A6).  Fully masked KV tiles are skipped before they are loaded.
 * stream: NULL = run on the context stream and block until done (like every reference entry point);
 * non-NULL = a cudaStream_t; the call only enqueues, and q/k/v/out/lse/mask must be device-resident.
 * External masks are read in place (bool bytes, fp16 / bf16 / fp32; any broadcast; unit key stride for the tensor-core
 * kernels); a pre-pass leaves per-query-block lists of the KV tiles the mask keeps visible in context-owned scratch, so
 * enqueue-only calls that carry a mask (or quantised operands) must stay on ONE stream per context at a time. */
mfa_error_t mfa_attention_forward_ex(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t lse,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t window_size,
    mfa_precision_t input_precision, mfa_precision_t output_precision,
    const void* mask_ptr, size_t mask_size_bytes, const int64_t* mask_shape, const int64_t* mask_strides,
    uint32_t mask_ndim, mfa_mask_type_t mask_type, mfa_mask_scalar_t mask_scalar_type,
    void* stream);

/* One ring-attention step (SURVEY 8e; no reference counterpart): attention of seq_len_q query rows against a visiting
 * K/V block, merged in place -- L = log2(2^L_old + 2^L_new), O = O_old 2^(L_old-L) + O_new 2^(L_new-L) -- into rows
 * [acc_row_offset, acc_row_offset + seq_len_q) of every (b, h) of out_acc (fp32 [B,H,acc_rows,D]) and lse_acc
 * (fp32 [B,H,acc_rows], log2 units; rows holding -inf are simply overwritten).  bf16 / fp16 operands with head_dim 64 or
 * 128 only (MFA_ERROR_INVALID_ARGS otherwise); q / k / v may be strided handles; all buffers device-resident.
 * stream as in mfa_attention_forward_ex. */
mfa_error_t mfa_attention_forward_accumulate(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out_acc, mfa_buffer_t lse_acc,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t window_size, mfa_precision_t input_precision,
    uint32_t acc_row_offset, uint32_t acc_rows, void* stream);

/* P V precision of the quantised tensor-core forward (int8 / int4 codes, head_dim 128): e4m3 P and V on the fp8 tensor pipe
 * (default: BASELINE.json config 3, "int8 Q K^T and fp8 P V") or bf16 P with V's codes widened exactly to bf16.  Process-wide;
 * MFA_TCQ_PV=bf16|fp8 in the environment sets the initial value.  MFA_PRECISION_FP8_E4M3 exists for this setter only. */
#define MFA_PRECISION_FP8_E4M3 5
mfa_error_t mfa_set_quantized_pv_precision(mfa_context_t context, int32_t precision);   /* MFA_PRECISION_BF16 or MFA_PRECISION_FP8_E4M3 */
int32_t mfa_get_quantized_pv_precision(mfa_context_t context);

/* ---- ring attention (context parallelism over the GPUs of one node; SURVEY 8e, no reference counterpart) ----------------
 * One process per GPU; the sequence is cut into 2 * world chunks, rank r owns chunks r and 2 * world - 1 - r (zig-zag) stored
 * next to each other: q / k / v are device-resident contiguous [B, H, 2 * chunk_rows, D] (low chunk first), bf16 or fp16,
 * head_dim 64 or 128, chunk_rows a multiple of 256; out fp32 [B, H, 2 * chunk_rows, D], lse fp32 [B, H, 2 * chunk_rows] (log2).
 * One attention launch per ring step, the partial (O, L) merged in the kernel epilogue; every visiting pair has its own slot and
 * step s exchanges directly with ranks r +- s over NVLink / NVSwitch (csrc/ring.cu). */
typedef struct mfa_ring_opaque* mfa_ring_t;
bool mfa_ring_transport_available(void);                                   /* libnccl could be loaded */
mfa_error_t mfa_ring_get_unique_id(void* id_out, size_t id_bytes);         /* 128-byte NCCL id: rank 0 makes it, the host distributes it */
/* collective (ncclCommInitRank); unique_id NULL = no NCCL communicator, the ring can only use the p2p transport */
mfa_error_t mfa_ring_create(mfa_context_t context, const void* unique_id, size_t id_bytes, int32_t rank, int32_t world_size,
                            mfa_ring_t* ring);
mfa_error_t mfa_ring_create_from_comm(mfa_context_t context, void* nccl_comm, int32_t rank, int32_t world_size,
                                      mfa_ring_t* ring);                   /* caller-owned ncclComm_t of the same libnccl */
void mfa_ring_destroy(mfa_ring_t ring);
uint64_t mfa_ring_launch_count(mfa_ring_t ring);
int32_t mfa_ring_transport(mfa_ring_t ring);                               /* 0 = NCCL send / recv, 1 = p2p (copy engines) */
/* p2p transport (copy engines push each K/V pair straight into the receiver's slot, stream memory operations order the
 * streams; no SM takes part in a hop): prepare allocates the slots for the largest problem to come, export fills a blob of
 * mfa_ring_handle_bytes() bytes (CUDA IPC handles), the host gathers the blobs of all ranks in rank order -- any channel -- and
 * import opens them.  From then on mfa_ring_attention_forward uses p2p (MFA_RING_TRANSPORT=nccl|p2p picks the default). */
size_t mfa_ring_handle_bytes(void);
mfa_error_t mfa_ring_prepare(mfa_ring_t ring, uint32_t batch_size, uint32_t chunk_rows, uint32_t num_heads, uint16_t head_dim);
mfa_error_t mfa_ring_export_handles(mfa_ring_t ring, void* blob_out, size_t blob_bytes);
mfa_error_t mfa_ring_import_handles(mfa_ring_t ring, const void* blobs, size_t bytes_per_rank);
/* collective; stream = cudaStream_t of the attention launches (NULL: an internal stream, the call blocks until O is ready) */
mfa_error_t mfa_ring_attention_forward(
    mfa_ring_t ring, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t lse,
    uint32_t batch_size, uint32_t chunk_rows, uint32_t num_heads, uint16_t head_dim, float softmax_scale,
    mfa_precision_t precision, void* stream);

/* Backward of the ring forward (collective; NCCL transport: the ring must own or have been given a communicator).  out / lse: the
 * forward's results of this rank; dout in `precision` [B, H, 2 * chunk_rows, D]; dq / dk / dv fp32 [B, H, 2 * chunk_rows, D],
 * overwritten.  Same rectangles as the forward; dQ accumulates locally, the dK / dV of a visiting pair go straight back to its owner. */
mfa_error_t mfa_ring_attention_backward(
    mfa_ring_t ring, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t lse, mfa_buffer_t dout,
    mfa_buffer_t dq, mfa_buffer_t dk, mfa_buffer_t dv,
    uint32_t batch_size, uint32_t chunk_rows, uint32_t num_heads, uint16_t head_dim, float softmax_scale,
    mfa_precision_t precision, void* stream);

/* Backward twin of the above (mask and window honoured; the reference's backward takes neither). */
mfa_error_t mfa_attention_backward_ex(
    mfa_context_t context,
    mfa_buffer_t dout, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t softmax_lse,
    mfa_buffer_t dq, mfa_buffer_t dk, mfa_buffer_t dv, mfa_buffer_t d_buffer,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t window_size, mfa_precision_t input_precision,
    const void* mask_ptr, size_t mask_size_bytes, const int64_t* mask_shape, const int64_t* mask_strides,
    uint32_t mask_ndim, mfa_mask_type_t mask_type, mfa_mask_scalar_t mask_scalar_type,
    void* stream);

/* Attention over num_seqs sequences packed along the sequence axis, without a dense mask.  cu_seqlens_q / cu_seqlens_k are
 * int32 [num_seqs + 1] offsets: 0, non-decreasing, ending at total_q / total_k.  Query row i of segment s sees key j only when j
 * lies in segment s; causal and window_size then apply to the offsets inside the segment (i' = i - cu_q[s], j' = j - cu_k[s]:
 * causal hides j' > i', the window hides i' > j' + window_size), so one call gives what one mfa_attention_forward_ex /
 * mfa_attention_backward_ex call per segment gives.  A row that sees no key gets O = 0, L = -inf and no gradient.
 * q is [1, num_heads, total_q, D], k / v [1, num_kv_heads, total_k, D] (strided handles give the [total, heads, D] layout);
 * num_kv_heads divides num_heads, 0 = num_heads.  lse fp32 [num_heads, total_q] (log2 units, may be NULL in the forward).
 * Backward: out fp32 and dout in input_precision, contiguous [num_heads, total_q, D]; dq fp32 [num_heads, total_q, D], dk / dv
 * fp32 [num_kv_heads, total_k, D], contiguous, overwritten; d_buffer as in mfa_attention_backward_ex.
 * Host-readable cu_seqlens (host or managed memory) are checked (MFA_ERROR_INVALID_ARGS when malformed); device-resident ones
 * are not read by the host, and the kernels clamp every bound they derive from them, so a malformed array gives wrong numbers
 * but no access out of bounds.  stream as in mfa_attention_forward_ex. */
mfa_error_t mfa_attention_forward_varlen(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t lse,
    mfa_buffer_t cu_seqlens_q, mfa_buffer_t cu_seqlens_k, uint32_t num_seqs, uint32_t total_q, uint32_t total_k,
    uint32_t num_heads, uint32_t num_kv_heads, uint16_t head_dim, float softmax_scale, bool causal, int32_t window_size,
    mfa_precision_t input_precision, mfa_precision_t output_precision, void* stream);

mfa_error_t mfa_attention_backward_varlen(
    mfa_context_t context, mfa_buffer_t dout, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    mfa_buffer_t softmax_lse, mfa_buffer_t dq, mfa_buffer_t dk, mfa_buffer_t dv, mfa_buffer_t d_buffer,
    mfa_buffer_t cu_seqlens_q, mfa_buffer_t cu_seqlens_k, uint32_t num_seqs, uint32_t total_q, uint32_t total_k,
    uint32_t num_heads, uint32_t num_kv_heads, uint16_t head_dim, float softmax_scale, bool causal, int32_t window_size,
    mfa_precision_t input_precision, void* stream);

/* Attention of seq_len_q new query tokens per sequence against that sequence's K/V cache (decode, speculative decode,
 * chunked prefill).  Forward only.
 * q is a [batch_size, num_heads, seq_len_q, D] view (strided handles give [B, Sq, H, D]); out has the same shape in
 * output_precision (fp32, bf16 or fp16, may be strided); lse fp32 [B, num_heads, seq_len_q] (log2 units) or NULL.
 * Contiguous cache (page_size == 0, block_table NULL): k_cache / v_cache are [B, num_kv_heads, cache_capacity, D] views (strided
 * handles give [B, cache_capacity, num_kv_heads, D]).  Paged cache (page_size > 0): k_cache / v_cache are contiguous
 * [num_pages, page_size, num_kv_heads, D] pools and block_table is int32 [B, cache_capacity / page_size], row-major: key j of
 * sequence b is row j % page_size of page block_table[b][j / page_size].  page_size is a multiple of 16 and divides
 * cache_capacity.
 * cache_seqlens is int32 [B]: L_b valid keys of sequence b, the seq_len_q new tokens included (the caller writes their K / V into
 * the cache first).  Query row s sits at position p = L_b - seq_len_q + s and sees key j < L_b iff (!causal || j <= p) &&
 * (window_size < 0 || p - j <= window_size) (bottom-right alignment).  A row that sees no key (L_b = 0, or L_b < seq_len_q under
 * causal) gets O = 0, L = -inf.  Cache rows past L_b are read as part of their 128-key tile and must hold finite values.
 * num_kv_heads divides num_heads (0 = num_heads), num_heads / num_kv_heads <= 128; bf16 / fp16 operands, head_dim a multiple of 8
 * up to 128.  Anything else returns MFA_ERROR_INVALID_ARGS.
 * Host-readable cache_seqlens / block_table (host or managed memory) are checked: lengths in [0, cache_capacity], page ids in
 * [0, num_pages).  Device-resident ones are not read by the host; the kernels clamp lengths to [0, cache_capacity] and page ids
 * to [0, num_pages), so malformed arrays give wrong numbers but no access out of bounds.
 * The keys of long caches are split over several work items whose partials a second kernel merges; how many depends on the
 * shape and the GPU only, never on the lengths, so results are deterministic.  With stream != NULL the call only enqueues work:
 * no host synchronisation, no host read of device memory, and no allocation once the context's scratch has been sized for the
 * shape by an earlier call.  Such a call can be captured in a CUDA graph and replayed with new cache_seqlens and cache contents;
 * make one call of the shape outside the capture first (during capture a call that would have to grow the scratch returns
 * MFA_ERROR_MEMORY_ALLOCATION).  A scratch block a graph has captured is never freed before the context: a later call that needs
 * more scratch gets a new block.  Replays and other calls on the context order themselves through an event, on any stream. */
mfa_error_t mfa_attention_forward_kvcache(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k_cache, mfa_buffer_t v_cache, mfa_buffer_t out, mfa_buffer_t lse,
    mfa_buffer_t cache_seqlens, mfa_buffer_t block_table,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t num_heads, uint32_t num_kv_heads, uint16_t head_dim,
    uint32_t cache_capacity, uint32_t page_size, uint32_t num_pages,
    float softmax_scale, bool causal, int32_t window_size,
    mfa_precision_t input_precision, mfa_precision_t output_precision, void* stream);

/* Device quantiser (GEMMQuantization.swift:305-623 / GEMMRuntimeQuantization.swift:80-181 contract):
 * src is a row-major [rows, cols] matrix of src_precision; scale[b] = absmax(block b) / 127 (int8) or / 7
 * (int4), floored at scale_floor when scale_floor > 0 (the reference GPU path uses 1e-8); codes =
 * clamp(round_half_away(x / scale)); int4 packs two codes per byte, element 2i in the low nibble, stored
 * +8.  Blocks are block_rows x block_cols tiles, scales row-major over blocks (0 = whole extent).
 * codes: rows*cols bytes (int8) or (rows*cols+1)/2 bytes (int4); scales: fp32 [n_blocks]. */
mfa_error_t mfa_quantize(
    mfa_context_t context, mfa_buffer_t src, mfa_buffer_t codes, mfa_buffer_t scales,
    uint64_t rows, uint64_t cols, uint32_t block_rows, uint32_t block_cols,
    mfa_precision_t src_precision, mfa_precision_t target_precision, float scale_floor, void* stream);

/* Inverse: out[i] = code[i] * scale[block(i)] as fp32. */
mfa_error_t mfa_dequantize(
    mfa_context_t context, mfa_buffer_t codes, mfa_buffer_t scales, mfa_buffer_t out,
    uint64_t rows, uint64_t cols, uint32_t block_rows, uint32_t block_cols,
    mfa_precision_t code_precision, void* stream);

/* Log-sum-exp merge of two partial attention results over disjoint key sets (ring attention step):
 *   L = log2(2^L_acc + 2^L_part);  O_acc = O_acc * 2^(L_acc - L) + O_part * 2^(L_part - L);  L_acc = L.
 * o_* fp32 [rows, head_dim], l_* fp32 [rows] (log2 units, the forward's L).  Rows with L_part = -inf are
 * left untouched. */
mfa_error_t mfa_merge_partials(
    mfa_context_t context, mfa_buffer_t o_acc, mfa_buffer_t l_acc, mfa_buffer_t o_part, mfa_buffer_t l_part,
    uint64_t rows, uint32_t head_dim, void* stream);

/* Device selection for one-process-per-GPU launches: must be called before the first mfa_create_context
 * in the process (the context is a singleton bound to one device).  Also honours MFA_CUDA_DEVICE. */
mfa_error_t mfa_set_device(int32_t device_index);
int32_t mfa_get_device_count(void);

/* Name of the kernel family the last compute call dispatched to ("fwd_tc_bf16_d128", "fwd_simt", ...);
 * static storage, do not free.  For tests and profiling only. */
const char* mfa_last_kernel_name(mfa_context_t context);

/* Number of kernels this library launched since the context was created (bench.py's gpu_launches). */
uint64_t mfa_launch_count(mfa_context_t context);

#ifdef __cplusplus
}
#endif

#endif /* MFA_FFI_EXT_H */
