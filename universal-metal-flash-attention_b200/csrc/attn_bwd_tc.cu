// attn_bwd_tc.cu -- attention backward for sm_100a on tcgen05 / TMEM / TMA (bf16 / fp16 operands, head_dim 64 / 128).
//
// Replaces the reference's two backward kernels (`loopBackwardKeyValue` / `loopBackwardQuery`,
// metal-flash-attention/Sources/FlashAttention/Attention/AttentionKernel/AttentionKernel+Source.swift:418-511, with the
// dS rule of +Softmax.swift:798-802 and the D term of +Softmax.swift:31-236) -- same 2-kernel split (no fp32 atomics,
// deterministic), re-derived for Blackwell:
//
//   bwd_dkv_tc_kernel : one CTA owns one 128-key tile j of one kv head and streams the query tiles i that can see it
//        S^T  = K_j Q_i^T            tcgen05.mma SS  -> TMEM cols [0,128)
//        dP^T = V_j dO_i^T           tcgen05.mma SS  -> TMEM cols [128,256)
//        P^T  = exp2(S^T c - L_i)    (two warpgroups, thread = (key row, 64-query half); 16-bit pairs back into TMEM)
//        dS^T = P^T (dP^T scale - D_i)
//        dV  += P^T  dO_i            tcgen05.mma TS (A from TMEM, B = dO_i tile read MN-major) -> cols [256,256+D)
//        dK  += dS^T Q_i             tcgen05.mma TS                                            -> cols [256+D,256+2D)
//   bwd_dq_tc_kernel  : one CTA owns one 128-query tile i and streams the key tiles j it can see
//        S = Q_i K_j^T (double-buffered in TMEM), dP = dO_i V_j^T, dS = P (dP scale - D_i), dQ += dS K_j (TS MMA)
//
// The MMA order is interleaved (dV_i, S^T_{i+1}, dK_i, dP^T_{i+1}) so the exp2 phase of tile i+1 runs under the
// dK_i / dP^T_{i+1} MMAs.  Packed P^T / dS^T are written inside the column range their owner thread read them from
// (half h reads fp32 cols [64h,64h+64) and writes 16-bit pairs to [64h,64h+32)), so the two warpgroups never touch
// each other's TMEM columns and need no cross-warpgroup barrier.
// Tiles fully hidden by the causal / sliding-window rule are skipped before they are loaded.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <math_constants.h>

#include "common.h"
#include "sm100_ptx.cuh"
#include "tc_host.h"

namespace mfa {

namespace {

using namespace ptx;

constexpr int kThreads = 384;     // warps 0-7: two elementwise warpgroups, 8: MMA issuer, 9: TMA, 10-11: L / D loaders
constexpr float kLog2e = 1.4426950408889634f;

struct BwdTcParams {
  CUtensorMap tq, tk, tv, tdo;
  CUtensorMap tdq, tdk, tdv;   // fp32 gradients, box = 32 floats x 128 rows (valid when g_tma != 0)
  int g_tma;                   // epilogues stage the gradients in shared memory and write them with TMA bulk stores
  const float* lse;
  const float* dterm;
  float* dq;
  float* dk;
  float* dv;
  int H, Hkv, Sq, Skv;
  float c, scale;
  int causal, window;
  // external mask (MASKED kernels): bool bytes (non-zero = attend) or additive values, element strides over [B,H,Sq,Skv]
  // with broadcast dims = 0 and unit key stride; P = exp2(S c + mask log2 e - L)
  const void* mask;
  int mask_kind, mask_scalar;
  long long mask_sb, mask_sh, mask_sq;
  // dense 1- / 2-byte masks: 128 x 128 tiles staged in shared memory by TMA (tm over [MB, MH, Sq, Skv], tc::make_mask_map)
  CUtensorMap tm;
  int mask_tma;
  // visible-tile lists under an external mask (null = walk the whole causal / window range):
  //   dQ kernel:  per (mask batch, mask head, 256-row query block) the KV tiles with a visible element   [lists][m_nkt]
  //   dK/dV kernel (H == Hkv only): per (mask batch, mask head, KV tile) the 128-row query tiles           [listsT][2 m_nqb]
  const int* ktiles; const int* kcounts;
  const int* qtiles; const int* qcounts;
  int m_nqb, m_nkt;
  const int* cu_q;             // packed variable-length sequences (AttnParams::cu_q / cu_k / nseq), or null
  const int* cu_k;
  int nseq;
};
constexpr int kTileNoMask = 1 << 30;          // list entry flag: the mask is a no-op on this tile (no loads needed)

// 32 mask terms in log2 units (-inf = hidden) for elements off0 + i * stride, i < nvalid (the rest: 0, they belong to dead
// rows / columns whose P is zeroed elsewhere).  The type switch sits outside the unrolled loops.
__device__ __forceinline__ void mask_terms32(const BwdTcParams& p, long long off0, long long stride, int nvalid, float* mt) {
  if (stride == 1 && nvalid == 32) {
    // row-owner layout (dQ kernel): 32 consecutive elements of one row -> 32-byte sector loads when aligned
    if (p.mask_kind == kMaskBool) {
      const uint8_t* m = reinterpret_cast<const uint8_t*>(p.mask) + off0;
      if ((reinterpret_cast<uintptr_t>(m) & 31) == 0) {
        uint32_t w[8];
        ldg256(m, w);
#pragma unroll
        for (int i = 0; i < 32; ++i) mt[i] = ((w[i >> 2] >> (8 * (i & 3))) & 0xffu) ? 0.f : -CUDART_INF_F;
        return;
      }
    } else if (p.mask_scalar == kMaskF32) {
      const float* m = reinterpret_cast<const float*>(p.mask) + off0;
      if ((reinterpret_cast<uintptr_t>(m) & 31) == 0) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t w[8];
          ldg256(m + 8 * c, w);
#pragma unroll
          for (int i = 0; i < 8; ++i) mt[8 * c + i] = __uint_as_float(w[i]) * kLog2e;
        }
        return;
      }
    } else {
      const uint16_t* m = reinterpret_cast<const uint16_t*>(p.mask) + off0;
      if ((reinterpret_cast<uintptr_t>(m) & 31) == 0) {
        const bool bf = p.mask_scalar == kMaskBF16;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t w[8];
          ldg256(m + 16 * c, w);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint32_t lo = w[i] & 0xffffu, hi = w[i] >> 16;
            mt[16 * c + 2 * i] = (bf ? __uint_as_float(lo << 16) : __half2float(__ushort_as_half((unsigned short)lo))) * kLog2e;
            mt[16 * c + 2 * i + 1] = (bf ? __uint_as_float(hi << 16) : __half2float(__ushort_as_half((unsigned short)hi))) * kLog2e;
          }
        }
        return;
      }
    }
  }
  // strided path (dK/dV kernel: one element per query row): two passes over the same registers -- first nothing but the 32
  // loads (raw bits parked in mt[]), then the conversions -- so all requests are in flight together.  (Fused into one loop the
  // compiler issued load, convert, load, convert ...: 64 serialised L2 round trips per step; profiles/r01n_ncu_full_dkv_masked.txt)
  if (p.mask_kind == kMaskBool) {
    const uint8_t* m = reinterpret_cast<const uint8_t*>(p.mask) + off0;
#pragma unroll
    for (int i = 0; i < 32; ++i) mt[i] = __uint_as_float(ldg_pred_u8(m + i * stride, i < nvalid, 1u));
#pragma unroll
    for (int i = 0; i < 32; ++i) mt[i] = __float_as_uint(mt[i]) == 0u ? -CUDART_INF_F : 0.f;
  } else if (p.mask_scalar == kMaskF32) {
    const float* m = reinterpret_cast<const float*>(p.mask) + off0;
#pragma unroll
    for (int i = 0; i < 32; ++i) mt[i] = __uint_as_float(ldg_pred_b32(m + i * stride, i < nvalid, 0u));
#pragma unroll
    for (int i = 0; i < 32; ++i) mt[i] *= kLog2e;
  } else {
    const uint16_t* m = reinterpret_cast<const uint16_t*>(p.mask) + off0;
    const bool bf = p.mask_scalar == kMaskBF16;
#pragma unroll
    for (int i = 0; i < 32; ++i) mt[i] = __uint_as_float(ldg_pred_u16(m + i * stride, i < nvalid, 0u));
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const uint32_t raw = __float_as_uint(mt[i]);
      mt[i] = (bf ? __uint_as_float(raw << 16) : __half2float(__ushort_as_half((unsigned short)raw))) * kLog2e;
    }
  }
}

template <int D, bool STAGED = false>
struct BCfg {
  static constexpr int kTile = 128 * D * 2;
  static constexpr int kChunks = D / 64;
  static constexpr int kChunkBytes = 128 * 128;
  // ring depths: A = operand used last (Q / K), B = dO / V.  STAGED (external mask tiles in shared memory): the 32 KB mask tile
  // takes the place of the second B stage at D = 128 (dO_i / V_j have one reader group per step and a whole step to reload)
#if defined(MFA_BWD_RA) && defined(MFA_BWD_RB)                  // ring-depth experiments (unmasked kernels, D = 128)
  static constexpr int kRA = (!STAGED && D == 128) ? MFA_BWD_RA : 3, kRB = (STAGED && D == 128) ? 1 : (D == 128 ? MFA_BWD_RB : 2);
#else
  static constexpr int kRA = 3, kRB = (STAGED && D == 128) ? 1 : 2;
#endif
  static constexpr int kMaskBytes = STAGED ? 128 * 128 * 2 : 0;  // one 128 x 128 tile of 16-bit terms (bool bytes use half)
  static constexpr int kStatBytes = 2 * 2 * 128 * 4;             // [slot][L|D][128], own 2-deep ring
  static constexpr int kSmem = (2 + kRA + kRB) * kTile + kMaskBytes + kStatBytes + 256 + 512;   // D = 128: 232192 of 232448 B
  static_assert(kSmem <= 232448, "shared memory budget of one CTA");
};

// Mask terms (log2 units, -inf = hidden) of one staged tile.  The tile sits in shared memory as TMA delivered it: rows = queries,
// 128 bytes of keys per row and chunk (16-bit terms: two chunks of 64 keys, 16 KB apart; bool bytes: one chunk of 128 keys),
// 16-byte unit j of row r at j ^ (r & 7).
// row-owner read (dQ kernel): the 64 keys [64 half, 64 half + 64) of query row `row`
__device__ __forceinline__ void staged_terms_row(const BwdTcParams& p, uint32_t tile, int row, int half, float* mt) {
  const uint32_t sw = (uint32_t)(row & 7);
  if (p.mask_kind == kMaskBool) {
    const uint32_t line = tile + (uint32_t)row * 128u;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float f0, f1, f2, f3;
      ptx::ld_shared_v4(line + (((uint32_t)(4 * half + j) ^ sw) << 4), f0, f1, f2, f3);
      const uint32_t w4[4] = {__float_as_uint(f0), __float_as_uint(f1), __float_as_uint(f2), __float_as_uint(f3)};
#pragma unroll
      for (int k = 0; k < 16; ++k) mt[16 * j + k] = ((w4[k >> 2] >> (8 * (k & 3))) & 0xffu) ? 0.f : -CUDART_INF_F;
    }
  } else {
    const uint32_t line = tile + (uint32_t)half * 16384u + (uint32_t)row * 128u;
    const bool bf = p.mask_scalar == kMaskBF16;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float f0, f1, f2, f3;
      ptx::ld_shared_v4(line + (((uint32_t)j ^ sw) << 4), f0, f1, f2, f3);
      const uint32_t w4[4] = {__float_as_uint(f0), __float_as_uint(f1), __float_as_uint(f2), __float_as_uint(f3)};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float lo, hi;
        if (bf) { lo = __uint_as_float(w4[k] << 16); hi = __uint_as_float(w4[k] & 0xffff0000u); }
        else { const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w4[k])); lo = f.x; hi = f.y; }
        mt[8 * j + 2 * k] = lo * kLog2e;
        mt[8 * j + 2 * k + 1] = hi * kLog2e;
      }
    }
  }
}
// column-owner read (dK/dV kernel): key column `col` of the 64 query rows [64 half, 64 half + 64); the 32 lanes of a warp read 32
// neighbouring keys of one row per request (64 or 32 consecutive bytes: no bank conflicts)
__device__ __forceinline__ void staged_terms_col(const BwdTcParams& p, uint32_t tile, int col, int half, float* mt) {
  if (p.mask_kind == kMaskBool) {
    const uint32_t unit = (uint32_t)(col >> 4), byte = (uint32_t)(col & 15);
#pragma unroll
    for (int i = 0; i < 64; ++i) {
      const uint32_t q = (uint32_t)(64 * half + i);
      mt[i] = ptx::ld_shared_u8(tile + q * 128u + ((unit ^ (q & 7u)) << 4) + byte) ? 0.f : -CUDART_INF_F;
    }
  } else {
    const uint32_t chunk = tile + (uint32_t)(col >> 6) * 16384u;
    const uint32_t unit = (uint32_t)((col & 63) >> 3), byte = (uint32_t)(col & 7) * 2u;
    const bool bf = p.mask_scalar == kMaskBF16;
#pragma unroll
    for (int i = 0; i < 64; ++i) {
      const uint32_t q = (uint32_t)(64 * half + i);
      const uint32_t raw = ptx::ld_shared_u16(chunk + q * 128u + ((unit ^ (q & 7u)) << 4) + byte);
      mt[i] = (bf ? __uint_as_float(raw << 16) : __half2float(__ushort_as_half((unsigned short)raw))) * kLog2e;
    }
  }
}


__device__ __forceinline__ void load_tile_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int row, int head, int b,
                                             int chunks, int chb) {
  for (int ch = 0; ch < chunks; ++ch) tma_load_4d(dst + ch * chb, m, bar, ch * 64, row, head, b);
}

// ================================================================================================ dK / dV
template <int D, bool BF16, int MASKED = 0>      // MASKED: 0 no external mask, 1 read in place, 2 tiles staged by TMA
__global__ void __launch_bounds__(kThreads, 1) bwd_dkv_tc_kernel(const __grid_constant__ BwdTcParams p) {
  using C = BCfg<D, MASKED == 2>;
  constexpr bool MT = MASKED == 2;
  constexpr int TILE = C::kTile, CHB = C::kChunkBytes;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  const uint32_t sK = base, sV = base + TILE;
  constexpr int RA = C::kRA, RB = C::kRB;
  auto sQ = [&](int s) { return base + (2 + s) * TILE; };            // ring A: Q_i (read by S^T_i first, dK_i last)
  auto sdO = [&](int s) { return base + (2 + RA + s) * TILE; };      // ring B: dO_i (dP^T_i, dV_i)
  const uint32_t sMask = base + (2 + RA + RB) * TILE;                // MT: the staged mask tile of the current step
  const uint32_t sStat = sMask + C::kMaskBytes;
  float* stat = reinterpret_cast<float*>(smem_raw + (sStat - raw));     // [stage][0: L, 1: D][128]
  const uint32_t sBar = sStat + C::kStatBytes;
  const uint32_t kv_full = sBar, s_full = sBar + 8, dp_full = sBar + 16, p_full = sBar + 24, ds_full = sBar + 32,
                 acc_full = sBar + 40;
  auto q_full = [&](int s) { return sBar + 48 + 8 * s; };
  auto q_empty = [&](int s) { return sBar + 80 + 8 * s; };
  auto do_full = [&](int s) { return sBar + 112 + 8 * s; };
  auto do_empty = [&](int s) { return sBar + 128 + 8 * s; };
  auto stat_full = [&](int s) { return sBar + 144 + 8 * s; };
  auto stat_empty = [&](int s) { return sBar + 160 + 8 * s; };
  const uint32_t tmem_slot = sBar + 176;
  const uint32_t mk_full = sBar + 184, mk_empty = sBar + 192;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp-uniform for ptxas
  // packed variable-length sequences (common.h): unmasked instantiations only -- segments do not combine with external masks
  const int* const seg_q = MASKED ? nullptr : p.cu_q;
  const int* const seg_k = MASKED ? nullptr : p.cu_k;
  const int jt = blockIdx.x, hk = blockIdx.y, b = blockIdx.z;
  const int c0 = jt * 128;
  const int group = p.H / p.Hkv;
  int qlo, qhi;
  block_query_range(p.causal, p.window, p.Sq, p.Skv, seg_q, seg_k, p.nseq, c0, min(c0 + 128, p.Skv), qlo, qhi);
  const int i_lo = qlo >> 7;
  int nq = qhi > qlo ? ((qhi + 127) >> 7) - i_lo : 0;
  const int* qlist = nullptr;                 // visible query tiles of this KV tile under the external mask
  if constexpr (MASKED) {
    if (p.qtiles) {
      const int lid = ((p.mask_sb ? b : 0) * (p.mask_sh ? p.H : 1) + (p.mask_sh ? hk : 0)) * p.m_nkt + jt;
      qlist = p.qtiles + (size_t)lid * (2 * p.m_nqb);
      nq = __ldg(p.qcounts + lid);
    }
  }
  const int n_it = nq * group;
  auto qtile_of = [&](int it) { return qlist ? (__ldg(qlist + it) & (kTileNoMask - 1)) : i_lo + it % nq; };

  if (threadIdx.x == 256) {
    mbar_init(kv_full, 1); mbar_init(s_full, 1); mbar_init(dp_full, 1); mbar_init(p_full, 8); mbar_init(ds_full, 8);
    mbar_init(acc_full, 1);
    for (int s = 0; s < RA; ++s) { mbar_init(q_full(s), 1); mbar_init(q_empty(s), 1); }
    for (int s = 0; s < RB; ++s) { mbar_init(do_full(s), 1); mbar_init(do_empty(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(stat_full(s), 2); mbar_init(stat_empty(s), 8); }
    if constexpr (MT) { mbar_init(mk_full, 1); mbar_init(mk_empty, 8); }
    fence_mbar_init();
  }
  if (warp == 9) {
    if (lane == 0) { prefetch_tmap(&p.tq); prefetch_tmap(&p.tk); prefetch_tmap(&p.tv); prefetch_tmap(&p.tdo); }
    __syncwarp();
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw)), 0);
  constexpr uint32_t T_S = 0, T_DP = 128, T_DV = 256, T_DK = 256 + D;

  if (warp == 9) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0 && n_it > 0) {
      mbar_arrive_expect_tx(kv_full, 2 * TILE);
      load_tile_4d(sK, &p.tk, kv_full, c0, hk, b, C::kChunks, CHB);
      load_tile_4d(sV, &p.tv, kv_full, c0, hk, b, C::kChunks, CHB);
      int mc = 0;                                        // staged mask tiles requested
      for (int it = 0; it < n_it; ++it) {
        const int sa = it % RA, sb = it % RB;
        const int head = hk * group + it / nq, q0 = qtile_of(it) * 128;
        mbar_wait(q_empty(sa), ((it / RA) & 1) ^ 1);
        mbar_arrive_expect_tx(q_full(sa), TILE);
        load_tile_4d(sQ(sa), &p.tq, q_full(sa), q0, head, b, C::kChunks, CHB);
        if constexpr (MT) {
          // mask tile [queries of Q_i] x [this CTA's keys]: its buffer is free once the elementwise warps have read the previous
          // one (at the start of their step), a whole step before this one is needed
          if (!(qlist && (__ldg(qlist + it) & kTileNoMask))) {
            if (mc > 0) mbar_wait(mk_empty, (mc - 1) & 1);
            const int mh = p.mask_sh ? head : 0, mb = p.mask_sb ? b : 0;
            if (p.mask_kind == kMaskBool) {
              mbar_arrive_expect_tx(mk_full, 16384);
              tma_load_4d(sMask, &p.tm, mk_full, c0, q0, mh, mb);
            } else {
              mbar_arrive_expect_tx(mk_full, 32768);
              tma_load_4d(sMask, &p.tm, mk_full, c0, q0, mh, mb);
              tma_load_4d(sMask + 16384, &p.tm, mk_full, c0 + 64, q0, mh, mb);
            }
            ++mc;
          }
        }
        mbar_wait(do_empty(sb), ((it / RB) & 1) ^ 1);
        mbar_arrive_expect_tx(do_full(sb), TILE);
        load_tile_4d(sdO(sb), &p.tdo, do_full(sb), q0, head, b, C::kChunks, CHB);
      }
    }
  } else if (warp >= 10) {
    // ------------------------------------------------------------------ L / D loaders (64 threads, 2 rows each)
    const int tl = threadIdx.x - 320;
    for (int it = 0; it < n_it; ++it) {
      const int s = it & 1;
      const int head = hk * group + it / nq, q0 = qtile_of(it) * 128;
      mbar_wait(stat_empty(s), ((it >> 1) & 1) ^ 1);
      const size_t rb = ((size_t)b * p.H + head) * p.Sq;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int r = tl + 64 * k, q = q0 + r;
        float L = CUDART_INF_F, Dt = 0.f;
        if (q < p.Sq) {
          L = p.lse[rb + q]; Dt = p.dterm[rb + q];
          if (L == -CUDART_INF_F) L = CUDART_INF_F;          // row without visible keys: P = 0
        }
        stat[(s * 2 + 0) * 128 + r] = L;
        stat[(s * 2 + 1) * 128 + r] = Dt;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(stat_full(s));
    }
  } else if (warp == 8) {
    // ------------------------------------------------------------------ MMA issuer (whole warp, elected lane issues)
    if (n_it > 0) {
      constexpr uint32_t FMT = BF16 ? 1u : 0u;
      constexpr uint32_t IDESC_ST = make_idesc(1, FMT, FMT, 0, 0, 128, 128);   // K-major A and B
      constexpr uint32_t IDESC_ACC = make_idesc(1, FMT, FMT, 0, 1, 128, D);    // A from TMEM, B MN-major
      const uint32_t k_lo = desc_lo(sK, 16), v_lo = desc_lo(sV, 16);
      const uint32_t qk_lo = desc_lo(sQ(0), 16), dok_lo = desc_lo(sdO(0), 16);       // K-major views of the stage tiles
      const uint32_t qm_lo = desc_lo(sQ(0), CHB), dom_lo = desc_lo(sdO(0), CHB);     // MN-major views
      constexpr uint32_t STG = TILE >> 4;                                            // ring-slot stride in descriptor units
      auto issue_abt = [&](uint32_t dcol, uint32_t a0, uint32_t b0) {                // D = A B^T over head_dim
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk) {
          const uint32_t off = ((kk >> 2) * CHB + (kk & 3) * 32) >> 4;
          mma_f16_ss_u(tmem + dcol, a0 + off, kDescHiSw128, b0 + off, kDescHiSw128, IDESC_ST, kk > 0);
        }
      };
      auto issue_acc = [&](uint32_t dcol, uint32_t acol, uint32_t b0, bool acc) {    // D += A(tmem) B over 128 queries
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          mma_f16_ts_u(tmem + dcol, tmem + acol + (kk >> 2) * 64 + (kk & 3) * 8, b0 + kk * (2048 >> 4), kDescHiSw128,
                       IDESC_ACC, (acc || kk > 0) ? 1u : 0u);
      };
      mbar_wait(kv_full, 0);
      mbar_wait(q_full(0), 0);
      tc_fence_after();
      issue_abt(T_S, k_lo, qk_lo);
      tc_commit_u(s_full);
      mbar_wait(do_full(0), 0);
      tc_fence_after();
      issue_abt(T_DP, v_lo, dok_lo);
      tc_commit_u(dp_full);
      for (int it = 0; it < n_it; ++it) {
        const uint32_t sa = it % RA, sb = it % RB, na = (it + 1) % RA, nb = (it + 1) % RB;
        mbar_wait(p_full, it & 1);
        tc_fence_after();
        issue_acc(T_DV, T_S, dom_lo + sb * STG, it > 0);
        tc_commit_u(do_empty(sb));                       // dO_i: dP^T_i and dV_i were its only readers
        if (it + 1 < n_it) {
          mbar_wait(q_full(na), ((it + 1) / RA) & 1);
          tc_fence_after();
          issue_abt(T_S, k_lo, qk_lo + na * STG);
          tc_commit_u(s_full);
        }
        mbar_wait(ds_full, it & 1);
        tc_fence_after();
        issue_acc(T_DK, T_DP, qm_lo + sa * STG, it > 0);
        tc_commit_u(q_empty(sa));                        // Q_i (and its L / D rows): last reader was dK_i
        if (it + 1 < n_it) {
          mbar_wait(do_full(nb), ((it + 1) / RB) & 1);
          tc_fence_after();
          issue_abt(T_DP, v_lo, dok_lo + nb * STG);
          tc_commit_u(dp_full);
        }
      }
      tc_commit_u(acc_full);
    }
  } else {
    // ------------------------------------------------------------------ elementwise warpgroups
    const int half = warp >> 2, w = warp & 3;
    const int row = w * 32 + lane;
    const int key = c0 + row;
    const uint32_t lane_base = (uint32_t)(w * 32) << 16;
    const uint32_t tS = tmem + lane_base + T_S + half * 64;
    const uint32_t tDP = tmem + lane_base + T_DP + half * 64;
    const float c = p.c, scale = p.scale;
    int qlo_r, qhi_r;                                      // queries visible to this key: [qlo_r, qhi_r]
    key_query_range(p.causal, p.window, p.Sq, p.Skv, seg_q, seg_k, p.nseq, key, qlo_r, qhi_r);
    --qhi_r;
    int mkc = 0;                                           // staged mask tiles consumed
    for (int it = 0; it < n_it; ++it) {
      const int s = it & 1;
      const int q0 = qtile_of(it) * 128 + half * 64;
      const float* sL = stat + (s * 2 + 0) * 128 + half * 64;
      const float* sD = stat + (s * 2 + 1) * 128 + half * 64;
      // queries visible to this key: [qlo_r, qhi_r]; rows past Sq carry L = +inf (P = 0)
      const bool any_mask = __any_sync(0xffffffffu, q0 < qlo_r || q0 + 63 > qhi_r);
      const int lo_i = qlo_r - q0, hi_i = qhi_r - q0;
      float pv[64];
      if constexpr (MASKED) {
        // the mask terms of this (query tile, key) pair do not depend on S: they are requested before the wait for S and land
        // in the registers that will hold P (free at this point), so their latency hides under the MMA
        if (qlist && (__ldg(qlist + it) & kTileNoMask)) {          // the mask is a no-op on this tile: nothing to load
#pragma unroll
          for (int i = 0; i < 64; ++i) pv[i] = 0.f;
        } else if constexpr (MT) {
          // staged tile: rows past Sq / keys past Skv arrive as zeros (bool: hidden; additive: + 0 on rows whose L is +inf)
          mbar_wait(mk_full, mkc & 1);
          ++mkc;
          staged_terms_col(p, sMask, row, half, pv);
          __syncwarp();
          if (lane == 0) mbar_arrive(mk_empty);
        } else {
          const int head = hk * group + it / nq;
#pragma unroll
          for (int ch = 0; ch < 2; ++ch) {
            // mask[q][key] for 32 queries: consecutive lanes = consecutive keys, so every load is coalesced
            const int qa = q0 + ch * 32;
            const long long off = (long long)b * p.mask_sb + (long long)head * p.mask_sh + (long long)qa * p.mask_sq + min(key, p.Skv - 1);
            mask_terms32(p, off, p.mask_sq, key < p.Skv ? min(32, p.Sq - qa) : 0, pv + ch * 32);
          }
        }
      }
      mbar_wait(stat_full(s), (it >> 1) & 1);
      mbar_wait(s_full, it & 1);
      tc_fence_after();
#pragma unroll
      for (int ch = 0; ch < 2; ++ch) {
        uint32_t su[32];
        tmem_ld_x32(tS + ch * 32, su);
        const float* mt = pv + ch * 32;           // MASKED: mask terms loaded above; overwritten by P below
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 L4 = *reinterpret_cast<const float4*>(sL + ch * 32 + i);
          const float Ls[4] = {L4.x, L4.y, L4.z, L4.w};
#pragma unroll
          for (int k = 0; k < 4; ++k)
            pv[ch * 32 + i + k] = ex2(fmaf(__uint_as_float(su[i + k]), c, MASKED ? mt[i + k] - Ls[k] : -Ls[k]));
        }
        if (any_mask) {
#pragma unroll
          for (int i = 0; i < 32; ++i) pv[ch * 32 + i] = (ch * 32 + i < lo_i || ch * 32 + i > hi_i) ? 0.f : pv[ch * 32 + i];
        }
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 16; ++i)
          pk[i] = BF16 ? pack_bf16(pv[ch * 32 + 2 * i], pv[ch * 32 + 2 * i + 1]) : pack_f16(pv[ch * 32 + 2 * i], pv[ch * 32 + 2 * i + 1]);
        tmem_st_x16(tS + ch * 16, pk);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);

      mbar_wait(dp_full, it & 1);
      tc_fence_after();
#pragma unroll
      for (int ch = 0; ch < 2; ++ch) {
        uint32_t du[32];
        tmem_ld_x32(tDP + ch * 32, du);
        tmem_wait_ld();
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 D4 = *reinterpret_cast<const float4*>(sD + ch * 32 + i);
          const float Ds[4] = {D4.x, D4.y, D4.z, D4.w};
          float ds[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) ds[k] = pv[ch * 32 + i + k] * fmaf(__uint_as_float(du[i + k]), scale, -Ds[k]);
          pk[i / 2] = BF16 ? pack_bf16(ds[0], ds[1]) : pack_f16(ds[0], ds[1]);
          pk[i / 2 + 1] = BF16 ? pack_bf16(ds[2], ds[3]) : pack_f16(ds[2], ds[3]);
        }
        tmem_st_x16(tDP + ch * 16, pk);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { mbar_arrive(ds_full); mbar_arrive(stat_empty(s)); }
    }
    // ---------------------------------------------------------------- epilogue: dV, dK (fp32) -> global
    if (n_it > 0) {
      mbar_wait(acc_full, 0);
      tc_fence_after();
    }
    const bool live = key < p.Skv;
    const size_t orow = (((size_t)b * p.Hkv + hk) * p.Skv + key) * D + half * (D / 2);
#pragma unroll
    for (int which = 0; which < 2; ++which) {
      float* dst_base = which == 0 ? p.dv : p.dk;
      const uint32_t tA = tmem + lane_base + (which == 0 ? T_DV : T_DK) + half * (D / 2);
#pragma unroll
      for (int ch = 0; ch < D / 64; ++ch) {
        uint32_t ou[32];
        if (n_it > 0) {
          tmem_ld_x32(tA + ch * 32, ou);
          tmem_wait_ld();
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) ou[i] = 0u;
        }
        if (p.g_tma && dst_base) {
          // swizzled staging chunk in the operand memory (every MMA has retired): 32 columns of this key row = one 128-byte line
          const uint32_t line = base + (uint32_t)(which * (D / 32) + half * (D / 64) + ch) * (128u * 128u) + (uint32_t)row * 128u;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            st_shared_v4(line + (uint32_t)((i ^ (row & 7)) << 4), __uint_as_float(ou[4 * i]), __uint_as_float(ou[4 * i + 1]),
                         __uint_as_float(ou[4 * i + 2]), __uint_as_float(ou[4 * i + 3]));
        } else if (live && dst_base) {
          float* dst = dst_base + orow + ch * 32;
          if ((reinterpret_cast<uintptr_t>(dst) & 31) == 0) {       // one 32-byte sector per store: half the LSU requests
#pragma unroll
            for (int i = 0; i < 4; ++i) st_global_v8(dst + 8 * i, reinterpret_cast<const float*>(ou) + 8 * i);
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              reinterpret_cast<float4*>(dst)[i] = make_float4(__uint_as_float(ou[4 * i]), __uint_as_float(ou[4 * i + 1]),
                                                              __uint_as_float(ou[4 * i + 2]), __uint_as_float(ou[4 * i + 3]));
          }
        }
      }
    }
    if (p.g_tma) {
      fence_proxy_async_smem();
      named_bar_sync(1 + half, 128);
      if ((threadIdx.x & 127) == 0) {
#pragma unroll
        for (int which = 0; which < 2; ++which) {
          if ((which == 0 ? p.dv : p.dk) == nullptr) continue;
#pragma unroll
          for (int ch = 0; ch < D / 64; ++ch)
            tma_store_4d(which == 0 ? &p.tdv : &p.tdk, base + (uint32_t)(which * (D / 32) + half * (D / 64) + ch) * (128u * 128u),
                         half * (D / 2) + ch * 32, c0, hk, b);
        }
        bulk_commit();
        bulk_wait_read();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) tmem_dealloc(tmem, 512);
}

// ================================================================================================ dQ
template <int D, bool BF16, int MASKED = 0>
__global__ void __launch_bounds__(kThreads, 1) bwd_dq_tc_kernel(const __grid_constant__ BwdTcParams p) {
  using C = BCfg<D, MASKED == 2>;
  constexpr bool MT = MASKED == 2;
  constexpr int TILE = C::kTile, CHB = C::kChunkBytes;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  const uint32_t sQ = base, sdO = base + TILE;
  constexpr int RA = C::kRA, RB = C::kRB;
  auto sK = [&](int s) { return base + (2 + s) * TILE; };            // ring A: K_j (S_j first, dQ_j last)
  auto sV = [&](int s) { return base + (2 + RA + s) * TILE; };       // ring B: V_j (dP_j only)
  const uint32_t sMask = base + (2 + RA + RB) * TILE;                // MT: the staged mask tile of the current step
  const uint32_t sBar = sMask + C::kMaskBytes;
  const uint32_t q_full = sBar, dp_full = sBar + 8, ds_full = sBar + 16, acc_full = sBar + 24;
  auto s_full = [&](int u) { return sBar + 32 + 8 * u; };
  auto k_full = [&](int s) { return sBar + 48 + 8 * s; };
  auto k_empty = [&](int s) { return sBar + 80 + 8 * s; };
  auto v_full = [&](int s) { return sBar + 112 + 8 * s; };
  auto v_empty = [&](int s) { return sBar + 128 + 8 * s; };
  const uint32_t tmem_slot = sBar + 144;
  const uint32_t mk_full = sBar + 152, mk_empty = sBar + 160;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp-uniform for ptxas
  // packed variable-length sequences (common.h): unmasked instantiations only -- segments do not combine with external masks
  const int* const seg_q = MASKED ? nullptr : p.cu_q;
  const int* const seg_k = MASKED ? nullptr : p.cu_k;
  const int it_q = p.causal ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;     // heavy tiles first
  const int h = blockIdx.y, b = blockIdx.z;
  const int hk = h / (p.H / p.Hkv);
  const int r0 = it_q * 128;
  int klo, khi;
  block_key_range(p.causal, p.window, p.Sq, p.Skv, seg_q, seg_k, p.nseq, r0, min(r0 + 128, p.Sq), klo, khi);
  const int j_lo = klo >> 7;
  int n = khi > klo ? ((khi + 127) >> 7) - j_lo : 0;
  const int* klist = nullptr;                 // visible KV tiles of this tile's 256-row query block under the external mask
  if constexpr (MASKED) {
    if (p.ktiles) {
      const int lid = ((p.mask_sb ? b : 0) * (p.mask_sh ? p.H : 1) + (p.mask_sh ? h : 0)) * p.m_nqb + (it_q >> 1);
      klist = p.ktiles + (size_t)lid * p.m_nkt;
      n = __ldg(p.kcounts + lid);
    }
  }
  auto ktile_of = [&](int it) { return klist ? (__ldg(klist + it) & (kTileNoMask - 1)) : j_lo + it; };

  if (threadIdx.x == 256) {
    mbar_init(q_full, 1); mbar_init(dp_full, 1); mbar_init(ds_full, 8); mbar_init(acc_full, 1);
    for (int s = 0; s < 2; ++s) mbar_init(s_full(s), 1);
    for (int s = 0; s < RA; ++s) { mbar_init(k_full(s), 1); mbar_init(k_empty(s), 1); }
    for (int s = 0; s < RB; ++s) { mbar_init(v_full(s), 1); mbar_init(v_empty(s), 1); }
    if constexpr (MT) { mbar_init(mk_full, 1); mbar_init(mk_empty, 8); }
    fence_mbar_init();
  }
  if (warp == 9) {
    if (lane == 0) { prefetch_tmap(&p.tq); prefetch_tmap(&p.tk); prefetch_tmap(&p.tv); prefetch_tmap(&p.tdo); }
    __syncwarp();
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw)), 0);
  constexpr uint32_t T_DP = 256, T_DQ = 384;

  if (warp == 9) {
    if (lane == 0 && n > 0) {
      mbar_arrive_expect_tx(q_full, 2 * TILE);
      load_tile_4d(sQ, &p.tq, q_full, r0, h, b, C::kChunks, CHB);
      load_tile_4d(sdO, &p.tdo, q_full, r0, h, b, C::kChunks, CHB);
      int mc = 0;                                        // staged mask tiles requested
      for (int it = 0; it < n; ++it) {
        const int sa = it % RA, sb = it % RB;
        mbar_wait(k_empty(sa), ((it / RA) & 1) ^ 1);
        mbar_arrive_expect_tx(k_full(sa), TILE);
        load_tile_4d(sK(sa), &p.tk, k_full(sa), ktile_of(it) * 128, hk, b, C::kChunks, CHB);
        if constexpr (MT) {
          if (!(klist && (__ldg(klist + it) & kTileNoMask))) {       // mask tile [this CTA's queries] x [keys of K_j]
            if (mc > 0) mbar_wait(mk_empty, (mc - 1) & 1);
            const int mh = p.mask_sh ? h : 0, mb = p.mask_sb ? b : 0, kc0 = ktile_of(it) * 128;
            if (p.mask_kind == kMaskBool) {
              mbar_arrive_expect_tx(mk_full, 16384);
              tma_load_4d(sMask, &p.tm, mk_full, kc0, r0, mh, mb);
            } else {
              mbar_arrive_expect_tx(mk_full, 32768);
              tma_load_4d(sMask, &p.tm, mk_full, kc0, r0, mh, mb);
              tma_load_4d(sMask + 16384, &p.tm, mk_full, kc0 + 64, r0, mh, mb);
            }
            ++mc;
          }
        }
        mbar_wait(v_empty(sb), ((it / RB) & 1) ^ 1);
        mbar_arrive_expect_tx(v_full(sb), TILE);
        load_tile_4d(sV(sb), &p.tv, v_full(sb), ktile_of(it) * 128, hk, b, C::kChunks, CHB);
      }
    }
  } else if (warp == 8) {
    if (n > 0) {
      constexpr uint32_t FMT = BF16 ? 1u : 0u;
      constexpr uint32_t IDESC_ST = make_idesc(1, FMT, FMT, 0, 0, 128, 128);
      constexpr uint32_t IDESC_ACC = make_idesc(1, FMT, FMT, 0, 1, 128, D);
      const uint32_t q_lo = desc_lo(sQ, 16), do_lo = desc_lo(sdO, 16);
      const uint32_t kk_lo = desc_lo(sK(0), 16), vk_lo = desc_lo(sV(0), 16), km_lo = desc_lo(sK(0), CHB);
      constexpr uint32_t STG = TILE >> 4;
      auto issue_abt = [&](uint32_t dcol, uint32_t a0, uint32_t b0) {
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk) {
          const uint32_t off = ((kk >> 2) * CHB + (kk & 3) * 32) >> 4;
          mma_f16_ss_u(tmem + dcol, a0 + off, kDescHiSw128, b0 + off, kDescHiSw128, IDESC_ST, kk > 0);
        }
      };
      mbar_wait(q_full, 0);
      mbar_wait(k_full(0), 0);
      tc_fence_after();
      issue_abt(0, q_lo, kk_lo);
      tc_commit_u(s_full(0));
      mbar_wait(v_full(0), 0);
      tc_fence_after();
      issue_abt(T_DP, do_lo, vk_lo);
      tc_commit_u(dp_full);
      tc_commit_u(v_empty(0));
      for (int it = 0; it < n; ++it) {
        const uint32_t u = it & 1, sa = it % RA, na = (it + 1) % RA, nb = (it + 1) % RB;
        if (it + 1 < n) {
          mbar_wait(k_full(na), ((it + 1) / RA) & 1);
          tc_fence_after();
          issue_abt((u ^ 1) * 128, q_lo, kk_lo + na * STG);
          tc_commit_u(s_full(u ^ 1));
        }
        mbar_wait(ds_full, it & 1);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          mma_f16_ts_u(tmem + T_DQ, tmem + T_DP + (kk >> 2) * 64 + (kk & 3) * 8, km_lo + sa * STG + kk * (2048 >> 4),
                       kDescHiSw128, IDESC_ACC, (it > 0 || kk > 0) ? 1u : 0u);
        tc_commit_u(k_empty(sa));                        // K_j: S_j first, dQ_j last
        if (it + 1 < n) {
          mbar_wait(v_full(nb), ((it + 1) / RB) & 1);
          tc_fence_after();
          issue_abt(T_DP, do_lo, vk_lo + nb * STG);
          tc_commit_u(dp_full);
          tc_commit_u(v_empty(nb));                      // V_j is only read by dP_j
        }
      }
      tc_commit_u(acc_full);
    }
  } else if (warp < 8) {
    const int half = warp >> 2, w = warp & 3;
    const int row = w * 32 + lane;
    const int r = r0 + row;
    const uint32_t lane_base = (uint32_t)(w * 32) << 16;
    const uint32_t tDP = tmem + lane_base + T_DP + half * 64;
    const float c = p.c, scale = p.scale;
    float L = CUDART_INF_F, Dt = 0.f;
    if (r < p.Sq) {
      const size_t ri = ((size_t)b * p.H + h) * p.Sq + r;
      L = p.lse[ri]; Dt = p.dterm[ri];
      if (L == -CUDART_INF_F) L = CUDART_INF_F;
    }
    int clo, chi;                                          // visible keys of this row: [clo, chi]
    row_key_range(p.causal, p.window, p.Sq, p.Skv, seg_q, seg_k, p.nseq, r, clo, chi);
    --chi;
    int mkc = 0;                                           // staged mask tiles consumed
    for (int it = 0; it < n; ++it) {
      const int u = it & 1;
      const int k0 = ktile_of(it) * 128 + half * 64;
      const uint32_t tS = tmem + lane_base + u * 128 + half * 64;
      const bool any_mask = __any_sync(0xffffffffu, k0 < clo || k0 + 63 > chi);
      const int lo_i = clo - k0, hi_i = chi - k0;
      float pv[64];
      if constexpr (MASKED) {
        if (klist && (__ldg(klist + it) & kTileNoMask)) {
#pragma unroll
          for (int i = 0; i < 64; ++i) pv[i] = 0.f;
        } else if constexpr (MT) {
          mbar_wait(mk_full, mkc & 1);
          ++mkc;
          staged_terms_row(p, sMask, row, half, pv);
          __syncwarp();
          if (lane == 0) mbar_arrive(mk_empty);
        } else {
#pragma unroll
          for (int ch = 0; ch < 2; ++ch) {
            const int ka = k0 + ch * 32;
            const long long off = (long long)b * p.mask_sb + (long long)h * p.mask_sh + (long long)min(r, p.Sq - 1) * p.mask_sq + ka;
            mask_terms32(p, off, 1, r < p.Sq ? min(32, p.Skv - ka) : 0, pv + ch * 32);
          }
        }
      }
      mbar_wait(s_full(u), (it >> 1) & 1);
      tc_fence_after();
#pragma unroll
      for (int ch = 0; ch < 2; ++ch) {
        uint32_t su[32];
        tmem_ld_x32(tS + ch * 32, su);
        const float* mt = pv + ch * 32;           // MASKED: mask terms loaded above; overwritten by P below
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; ++i) pv[ch * 32 + i] = ex2(fmaf(__uint_as_float(su[i]), c, MASKED ? mt[i] - L : -L));
        if (any_mask) {
#pragma unroll
          for (int i = 0; i < 32; ++i) pv[ch * 32 + i] = (ch * 32 + i < lo_i || ch * 32 + i > hi_i) ? 0.f : pv[ch * 32 + i];
        }
      }
      mbar_wait(dp_full, it & 1);
      tc_fence_after();
#pragma unroll
      for (int ch = 0; ch < 2; ++ch) {
        uint32_t du[32];
        tmem_ld_x32(tDP + ch * 32, du);
        tmem_wait_ld();
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const float d0 = pv[ch * 32 + i] * fmaf(__uint_as_float(du[i]), scale, -Dt);
          const float d1 = pv[ch * 32 + i + 1] * fmaf(__uint_as_float(du[i + 1]), scale, -Dt);
          pk[i / 2] = BF16 ? pack_bf16(d0, d1) : pack_f16(d0, d1);
        }
        tmem_st_x16(tDP + ch * 16, pk);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(ds_full);
    }
    if (n > 0) {
      mbar_wait(acc_full, 0);
      tc_fence_after();
    }
    const bool live = r < p.Sq;
    const size_t orow = (((size_t)b * p.H + h) * p.Sq + r) * D + half * (D / 2);
    const uint32_t tA = tmem + lane_base + T_DQ + half * (D / 2);
#pragma unroll
    for (int ch = 0; ch < D / 64; ++ch) {
      uint32_t ou[32];
      if (n > 0) {
        tmem_ld_x32(tA + ch * 32, ou);
        tmem_wait_ld();
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) ou[i] = 0u;
      }
      if (p.g_tma) {
        const uint32_t line = base + (uint32_t)(half * (D / 64) + ch) * (128u * 128u) + (uint32_t)row * 128u;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          st_shared_v4(line + (uint32_t)((i ^ (row & 7)) << 4), __uint_as_float(ou[4 * i]), __uint_as_float(ou[4 * i + 1]),
                       __uint_as_float(ou[4 * i + 2]), __uint_as_float(ou[4 * i + 3]));
      } else if (live) {
        float* dst = p.dq + orow + ch * 32;
        if ((reinterpret_cast<uintptr_t>(dst) & 31) == 0) {
#pragma unroll
          for (int i = 0; i < 4; ++i) st_global_v8(dst + 8 * i, reinterpret_cast<const float*>(ou) + 8 * i);
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            reinterpret_cast<float4*>(dst)[i] = make_float4(__uint_as_float(ou[4 * i]), __uint_as_float(ou[4 * i + 1]),
                                                            __uint_as_float(ou[4 * i + 2]), __uint_as_float(ou[4 * i + 3]));
        }
      }
    }
    if (p.g_tma) {
      fence_proxy_async_smem();
      named_bar_sync(1 + half, 128);
      if ((threadIdx.x & 127) == 0) {
#pragma unroll
        for (int ch = 0; ch < D / 64; ++ch)
          tma_store_4d(&p.tdq, base + (uint32_t)(half * (D / 64) + ch) * (128u * 128u), half * (D / 2) + ch * 32, r0, h, b);
        bulk_commit();
        bulk_wait_read();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) tmem_dealloc(tmem, 512);
}

// ---- visible-tile lists for the backward, from the forward's tile flags (launch_mask_flags)
// dQ: same lists as the forward (KV tiles per 256-row query block).
__global__ void bwd_compact_k_kernel(const uint8_t* __restrict__ flags, int* __restrict__ tiles, int* __restrict__ counts,
                                     int lists, int nkt) {
  const int lid = blockIdx.x * blockDim.x + threadIdx.x;
  if (lid >= lists) return;
  int cnt = 0;
  for (int j = 0; j < nkt; ++j)
    if (const int f = flags[(size_t)lid * nkt + j]) tiles[(size_t)lid * nkt + cnt++] = j | (f == 2 ? kTileNoMask : 0);
  counts[lid] = cnt;
}
// dK/dV: per (mask batch x head, KV tile) the 128-row query tiles of every flagged 256-row block, clipped to the tile's own
// causal / window query range.
__global__ void bwd_compact_q_kernel(const uint8_t* __restrict__ flags, int* __restrict__ tiles, int* __restrict__ counts,
                                     int mbh_n, int nqb, int nkt, int Sq, int Skv, int causal, int window) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= mbh_n * nkt) return;
  const int mbh = idx / nkt, j = idx % nkt;
  int qlo, qhi;
  visible_query_range(causal, window, Sq, j * 128, min(j * 128 + 128, Skv), qlo, qhi);
  const int i_lo = qlo >> 7, i_hi = qhi > qlo ? (qhi + 127) >> 7 : i_lo;
  int cnt = 0;
  for (int qb = 0; qb < nqb; ++qb) {
    const int f = flags[((size_t)mbh * nqb + qb) * nkt + j];
    if (!f) continue;
    for (int t = 2 * qb; t < 2 * qb + 2; ++t)
      if (t >= i_lo && t < i_hi && t * 128 < Sq) tiles[(size_t)idx * (2 * nqb) + cnt++] = t | (f == 2 ? kTileNoMask : 0);
  }
  counts[idx] = cnt;
}

template <typename K>
cudaError_t ensure_smem(K kern, int bytes, bool& done) {
  if (done) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done = true;
  return e;
}

template <int D, bool BF16, int MASKED>
cudaError_t launch_bwd_m(const BwdTcParams& prm, int B, bool want_dq, bool want_dkv, cudaStream_t st) {
  static bool a_set = false, b_set = false;
  constexpr int kSmem = BCfg<D, MASKED == 2>::kSmem;
  cudaError_t e;
  if (want_dkv) {
    if ((e = ensure_smem(bwd_dkv_tc_kernel<D, BF16, MASKED>, kSmem, a_set)) != cudaSuccess) return e;
    dim3 grid((prm.Skv + 127) / 128, prm.Hkv, B);
    bwd_dkv_tc_kernel<D, BF16, MASKED><<<grid, kThreads, kSmem, st>>>(prm);
    ++g_launch_count;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  if (want_dq) {
    if ((e = ensure_smem(bwd_dq_tc_kernel<D, BF16, MASKED>, kSmem, b_set)) != cudaSuccess) return e;
    dim3 grid((prm.Sq + 127) / 128, prm.H, B);
    bwd_dq_tc_kernel<D, BF16, MASKED><<<grid, kThreads, kSmem, st>>>(prm);
    ++g_launch_count;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  return cudaSuccess;
}

template <int D, bool BF16>
cudaError_t launch_bwd(const BwdTcParams& prm, int B, bool want_dq, bool want_dkv, cudaStream_t st) {
  if (prm.mask && prm.mask_tma) return launch_bwd_m<D, BF16, 2>(prm, B, want_dq, want_dkv, st);
  return prm.mask ? launch_bwd_m<D, BF16, 1>(prm, B, want_dq, want_dkv, st)
                  : launch_bwd_m<D, BF16, 0>(prm, B, want_dq, want_dkv, st);
}

}  // namespace

bool bwd_tc_eligible(const AttnParams& p) {
  if (getenv("MFA_DISABLE_TC") || getenv("MFA_DISABLE_TC_BWD")) return false;
  if (p.in_dtype != kBF16 && p.in_dtype != kF16) return false;
  if (p.do_dtype != p.in_dtype) return false;
  // head dims 64 / 128 as they are; other multiples of 8 up to 128 on the next kernel width: TMA zero-fills the missing columns
  // of Q / K / V / dO and clips the gradient stores, so those need the TMA-store epilogues
  if (p.D < 8 || p.D > 128 || (p.D & 7)) return false;
  if (p.D != 64 && p.D != 128 && (getenv("MFA_DISABLE_TMA_STORE") || getenv("MFA_DISABLE_TC_PADDED_D"))) return false;
  if (p.mask_kind != kMaskNone && p.mask && (p.mask_sk != 1 || getenv("MFA_DISABLE_TC_MASK"))) return false;
  if (p.Sq <= 0 || p.Skv <= 0 || p.B <= 0 || p.H <= 0 || p.Hkv <= 0 || p.H % p.Hkv) return false;
  if (p.B > 65535 || p.H > 65535) return false;
  if (!tc::view_ok(p.q, p.H, p.B) || !tc::view_ok(p.k, p.Hkv, p.B) || !tc::view_ok(p.v, p.Hkv, p.B) ||
      !tc::view_ok(p.d_o, p.H, p.B))
    return false;
  if (!p.lse || !p.dterm) return false;
  for (float* g : {p.dq, p.dk, p.dv})
    if (g && (reinterpret_cast<uintptr_t>(g) & 15)) return false;
  return tc::encode_fn() != nullptr;
}

size_t bwd_tc_mask_scratch_bytes(const AttnParams& p) {
  if (p.mask_kind == kMaskNone || !p.mask || getenv("MFA_DISABLE_MASK_SKIP")) return 0;
  int nqb, nkt, MB, MH;
  mask_tile_dims(p, nqb, nkt, MB, MH);
  const size_t lists = (size_t)MB * MH * nqb, listsT = (size_t)MB * MH * nkt;
  if (lists > 0x3fffffffULL || listsT > 0x3fffffffULL) return 0;
  return (lists * (nkt + 1) + listsT * (2 * (size_t)nqb + 1)) * sizeof(int) + lists * nkt + 16;
}

// dQ, dK, dV from Q, K, V, dO, L and D (= scale * rowsum(dO * O), launch_dterm).  Gradients are fp32 contiguous BHSD.
cudaError_t launch_bwd_tc(const AttnParams& p, cudaStream_t st) {
  BwdTcParams prm;
  if (!tc::make_map(&prm.tq, p.q, p.in_dtype, p.B, p.H, p.Sq, p.D) ||
      !tc::make_map(&prm.tdo, p.d_o, p.in_dtype, p.B, p.H, p.Sq, p.D) ||
      !tc::make_map(&prm.tk, p.k, p.in_dtype, p.B, p.Hkv, p.Skv, p.D) ||
      !tc::make_map(&prm.tv, p.v, p.in_dtype, p.B, p.Hkv, p.Skv, p.D))
    return cudaErrorInvalidValue;
  prm.lse = p.lse; prm.dterm = p.dterm;
  prm.dq = p.dq; prm.dk = p.dk; prm.dv = p.dv;
  // gradients leave through swizzled staging tiles + TMA bulk stores (contiguous fp32 BHSD by contract)
  prm.g_tma = 0;
  if (!getenv("MFA_DISABLE_TMA_STORE")) {
    auto gview = [&](float* ptr, int Hn, int S) { return TensorView{ptr, (int64_t)Hn * S * p.D, (int64_t)S * p.D, (int64_t)p.D, 1}; };
    bool ok = true;
    if (p.dq) ok = ok && tc::make_map(&prm.tdq, gview(p.dq, p.H, p.Sq), kF32, p.B, p.H, p.Sq, p.D);
    if (p.dk) ok = ok && tc::make_map(&prm.tdk, gview(p.dk, p.Hkv, p.Skv), kF32, p.B, p.Hkv, p.Skv, p.D);
    if (p.dv) ok = ok && tc::make_map(&prm.tdv, gview(p.dv, p.Hkv, p.Skv), kF32, p.B, p.Hkv, p.Skv, p.D);
    prm.g_tma = ok ? 1 : 0;
  }
  prm.H = p.H; prm.Hkv = p.Hkv; prm.Sq = p.Sq; prm.Skv = p.Skv;
  prm.c = p.scale * kLog2e; prm.scale = p.scale;
  prm.causal = p.causal; prm.window = p.window;
  prm.cu_q = p.cu_q; prm.cu_k = p.cu_k; prm.nseq = p.nseq;
  prm.mask = nullptr; prm.mask_kind = kMaskNone; prm.mask_scalar = 0; prm.mask_sb = prm.mask_sh = prm.mask_sq = 0;
  if (p.mask_kind != kMaskNone && p.mask) {
    prm.mask = p.mask; prm.mask_kind = p.mask_kind; prm.mask_scalar = p.mask_scalar;
    prm.mask_sb = p.mask_sb; prm.mask_sh = p.mask_sh; prm.mask_sq = p.mask_sq;
  }
  prm.mask_tma = (prm.mask && tc::make_mask_map(&prm.tm, p)) ? 1 : 0;    // dense 1- / 2-byte masks: tiles staged by TMA
  prm.ktiles = prm.kcounts = prm.qtiles = prm.qcounts = nullptr; prm.m_nqb = prm.m_nkt = 0;
  cudaError_t e;
  if (prm.mask && p.mask_tile_scratch && bwd_tc_mask_scratch_bytes(p)) {
    int nqb, nkt, MB, MH;
    mask_tile_dims(p, nqb, nkt, MB, MH);
    const long long lists = (long long)MB * MH * nqb, listsT = (long long)MB * MH * nkt;
    int* kcounts = p.mask_tile_scratch;
    int* ktiles = kcounts + lists;
    int* qcounts = ktiles + lists * nkt;
    int* qtiles = qcounts + listsT;
    uint8_t* flags = reinterpret_cast<uint8_t*>(qtiles + listsT * 2 * nqb);
    if (launch_mask_flags(p, flags, st) == cudaSuccess) {
      bwd_compact_k_kernel<<<(unsigned)((lists + 127) / 128), 128, 0, st>>>(flags, ktiles, kcounts, (int)lists, nkt);
      prm.ktiles = ktiles; prm.kcounts = kcounts;
      if (p.H == p.Hkv) {            // grouped heads may carry different masks per head of a group: walk the full range
        bwd_compact_q_kernel<<<(unsigned)((listsT + 127) / 128), 128, 0, st>>>(flags, qtiles, qcounts, MB * MH, nqb, nkt, p.Sq,
                                                                             p.Skv, p.causal, p.window);
        prm.qtiles = qtiles; prm.qcounts = qcounts;
      }
      g_launch_count += 2;
      prm.m_nqb = nqb; prm.m_nkt = nkt;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    } else {
      cudaGetLastError();
    }
  }
  const bool want_dq = p.dq != nullptr, want_dkv = p.dk != nullptr && p.dv != nullptr;
  const bool bf = p.in_dtype == kBF16;
  const int Dk = p.D <= 64 ? 64 : 128;
  if (Dk != p.D && !prm.g_tma) return cudaErrorNotSupported;
  if (Dk == 128) e = bf ? launch_bwd<128, true>(prm, p.B, want_dq, want_dkv, st) : launch_bwd<128, false>(prm, p.B, want_dq, want_dkv, st);
  else e = bf ? launch_bwd<64, true>(prm, p.B, want_dq, want_dkv, st) : launch_bwd<64, false>(prm, p.B, want_dq, want_dkv, st);
  if (prm.mask && prm.mask_tma) g_last_kernel = Dk == 128 ? (bf ? "bwd_tc_bf16_d128_tma_mask" : "bwd_tc_fp16_d128_tma_mask") : (bf ? "bwd_tc_bf16_d64_tma_mask" : "bwd_tc_fp16_d64_tma_mask");
  else if (prm.mask) g_last_kernel = Dk == 128 ? (bf ? "bwd_tc_bf16_d128_mask" : "bwd_tc_fp16_d128_mask") : (bf ? "bwd_tc_bf16_d64_mask" : "bwd_tc_fp16_d64_mask");
  else g_last_kernel = Dk == 128 ? (bf ? "bwd_tc_bf16_d128" : "bwd_tc_fp16_d128") : (bf ? "bwd_tc_bf16_d64" : "bwd_tc_fp16_d64");
  return e;
}

}  // namespace mfa
