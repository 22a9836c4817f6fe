// attn_fwd_tc.cu -- fused attention forward for sm_100a: TMA -> shared memory -> tcgen05.mma -> TMEM.
//
// Replaces the reference's `attention` kernel, type = forward
// (metal-flash-attention/Sources/FlashAttention/Attention/AttentionKernel/AttentionKernel+Source.swift:372-416,
//  online softmax +Softmax.swift:641-702, finalisation +Caching.swift:396-400) for bf16/fp16 operands with
// head_dim 64 or 128, and -- operand mode kFwdI8 -- the quantised forward (QuantizedAttention.swift:71-91,358-463)
// for symmetric int8 codes at head_dim 128.  Same math, re-derived for Blackwell:
//
//   one CTA = 2 query tiles of 128 rows (one per softmax warpgroup) sharing one K/V stream
//   warp 9       : TMA producer   Q tiles once, then K_j, V_j tiles through an NS-stage mbarrier ring (128B swizzle)
//   warp 8 / 10  : MMA issuer of tile 0 / 1 (each tile has its own in-order chain, the tensor pipe interleaves them)
//                    S_t = Q_t K_j^T  (tcgen05.mma SS, fp32 -- or s32 for int8 codes -- accumulator in TMEM columns
//                                      [t*128, +128))
//                    O_t += P_t V_j   (tcgen05.mma TS: P read straight from TMEM, V MN-major from smem)
//   warps 0-3 / 4-7 : softmax warpgroup of tile 0 / 1; thread i owns row i of its tile (tcgen05.ld 32x32b), so
//                     row max / row sum need no shuffles; P is written back over S as packed 16-bit pairs.
//
// P is handed to the MMA warp in four 32-key parts: the P V MMAs of part k run while the softmax warps are still in
// exp2 on part k+1, so only the last quarter of P V and the next S sit on the per-tile dependency chain
// (ld S -> max -> exp2 -> P V -> S, which -- not pipe throughput -- bounds this kernel; profiles/).
// O is only rescaled when the running row max grew by more than 2^8 (the stale max is kept otherwise; the final
// division by l absorbs it), so the O read-modify-write in TMEM is rare.
// KV tiles that are fully hidden by the causal / sliding-window rule are never loaded (loop bounds), tiles that
// are partly hidden get an element mask, tiles that are fully visible skip the mask code.
// Outputs follow the reference contract: O fp32 (or fp16/bf16 on request) and L = m + log2(l) in log2 units.
//
// int8 mode: S_int = Q_i8 K_i8^T on kind::i8 (2x the bf16 MMA rate); the softmax warps widen it with I2FP (exact)
// and fold every scale into the one packed FFMA that forms the exponent:   x = s_int * a_h + (log2 v_h - m),   a_h = qs[row block] * ks[h] * scale * log2(e),
// h = 64-key half of the tile.  P' = P v_h (the V block scale rides in the exponent) feeds the P V MMA, which runs on
// kind::f16 with V's int8 codes widened to bf16 (exact); the row sum takes sum(P') / v_h per half.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <math_constants.h>

#include <algorithm>
#include <mutex>
#include <numeric>
#include <type_traits>

#include "common.h"
#include "fwd_tc.h"
#include "sm100_ptx.cuh"
#include "tc_host.h"

namespace mfa {

namespace {

using namespace ptx;

constexpr int kThreads = 384;           // warpgroups: softmax 0, softmax 1, {MMA 0, TMA, MMA 1, idle}
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr float kRescaleThreshold = 8.f;     // log2 units
constexpr int kTileNoMask = 1 << 30;          // flag bit in a visible-tile list entry
constexpr int kParts = 4;                    // P hand-off granularity: 32 keys = 16 packed TMEM columns

template <int D, int MODE, int MASKED = 0>      // MASKED: 0 no external mask, 1 read in place, 2 staged in shared memory
struct Cfg {
  static constexpr bool kI4 = MODE == kFwdI4 || MODE == kFwdI4F8;    // Q / K arrive as packed int4 and are unpacked in shared memory
  static constexpr bool kF8 = MODE == kFwdI8F8 || MODE == kFwdI4F8;  // int8 Q K^T, e4m3 P V
  static constexpr bool kI8 = MODE == kFwdI8 || kF8 || kI4;          // int8 Q K^T
  static constexpr bool kSplit = MODE == kFwdSplit;                  // fp32 operands as fp16 (hi, lo) pairs, 3 MMAs per product
  static constexpr bool kWide = MODE == kFwdWideF16 || MODE == kFwdWideBF16;   // head_dim 256: (a, b) halves of 128 columns
  static constexpr int kChunkBytes = 128 * 128;                      // one 128-byte swizzle chunk of 128 rows
  static constexpr int kQChunks = kI8 ? 1 : D / 64;                  // chunks per Q / K tile (split: per hi / lo half)
  static constexpr int kVChunks = kF8 ? 1 : D / 64;                  // V: 16-bit, or e4m3 (128 head dims = one 128-byte row)
  static constexpr int kHalf = kQChunks * kChunkBytes;               // one K tile, or one half (hi / lo) of a split tile
  static constexpr int kQTile = kHalf * ((kSplit || kWide) ? 2 : 1); // split: Q_hi then Q_lo; wide: Q_a then Q_b
  static constexpr int kVTile = kVChunks * kChunkBytes;
  static constexpr int kStage = kVTile;                              // ring stage (K tiles may use part of it)
  static constexpr int kSPS = kSplit ? 4 : kWide ? 3 : 2;            // ring stages per KV step (split: K_lo, K_hi, V_hi, V_lo; wide: K_a, K_b, V_half)
  // MASKED == 2 (16-bit operand modes only: the quantised entry points take fp32 masks): the external mask is staged in shared
  // memory, two 32 KB tiles fed by TMA (see the mask producer in warp 11).
  // Every masked kernel except the int4 ones runs on a shallow ring -- 96 KB instead of 160 KB: the unmasked kernel loses
  // nothing with it (0.216 vs 0.2145 ms, profiles/r02bb_*), the staged tiles need the room, and the in-place mask reads gain
  // 64 KB of L1 (dense fp32 [1, 1, S, S] mask: 0.58 -> 0.49 ms)
  static constexpr bool kMaskTma = MASKED == 2 && (MODE == kFwdF16 || MODE == kFwdBF16);
  static constexpr int kMaskTile = 128 * 128 * 2;                    // one query tile x 128 keys of 16-bit terms (bool bytes use half)
  static constexpr bool kShallow = MASKED != 0 && !kI4;
  static constexpr int kStages = (kSplit || kWide) ? 3               // split / wide: 2 x 64 KB of Q leave room for 3 x 32 KB
                               : (D == 128 && !kF8) ? (kShallow ? 3 : 5) : (kShallow ? 6 : 10);
  static constexpr int kBarBytes = 112 + 16 * kStages + 16 + 16 + 64 + 32; // + TMEM slot, o_empty, + raw-tile barriers (int4), + mask tile barriers
  // element pairs of every 8 whose exp2 runs on the FMA pipe (exp2_poly2) instead of MUFU.EX2; the fp32 split mode keeps exact
  // exp2 only (the polynomial's 8.6e-5 would show at fp32 tolerances)
  static constexpr int kPoly = kSplit ? 0 : 3;
  // int4: raw (packed) tiles as TMA delivers them -- a 3-deep ring of K tiles + one Q tile, 128 rows x 64 bytes each -- and
  // the per-row sums of the Q codes (2 x 128 ints)
  static constexpr int kRawTile = 128 * 64, kRawStages = 3;
  static constexpr int kRawBytes = kI4 ? (kRawStages + 1) * kRawTile + 1024 + 128 : 0;
  static constexpr int kMaskBytes = kMaskTma ? 2 * kMaskTile + 1024 : 0;
  static constexpr int kSmem = 2 * kQTile + kStages * kStage + kBarBytes + kRawBytes + kMaskBytes + 1024;
  static_assert(kSmem <= 232448, "shared memory budget of one CTA");
};

// 2^x for a pair of x <= ~8 on the FMA pipe (Cody-Waite split + degree-3 minimax polynomial, max rel err 8.6e-5),
// in packed f32x2 arithmetic: relieves the MUFU pipe, which is co-critical with the tensor pipe at head_dim 128
// (16 ex2/clk/SM vs 8192 FLOP/clk/SM).
__device__ __forceinline__ f32x2 exp2_poly2(f32x2 x) {
  float x0, x1;
  unpack2(x, x0, x1);
  // clamp at -127: a hidden element (x = -inf) gets r = -127, f = 0, p = 1.0 exactly, and 0x3F800000 + (-127 << 23) wraps to +0.0 --
  // an EXACT zero weight, so rows that are hidden completely keep l == 0; x in (-127, -126) gives a harmless denormal
  x = pack2(fmaxf(x0, -127.f), fmaxf(x1, -127.f));
  const f32x2 magic = pack2(12582912.f, 12582912.f);                  // 1.5 * 2^23: low mantissa bits = floor(x)
  const f32x2 xr = add2_rm(x, magic);
  const f32x2 f = sub2(x, sub2(xr, magic));                           // [0, 1)
  f32x2 pz = fma2(f, pack2(0.07706582f, 0.07706582f), pack2(0.22764632f, 0.22764632f));
  pz = fma2(pz, f, pack2(0.69511649f, 0.69511649f));
  pz = fma2(pz, f, pack2(1.0f, 1.0f));
  float p0, p1, r0, r1;
  unpack2(pz, p0, p1);
  unpack2(xr, r0, r1);
  return pack2(__int_as_float(__float_as_int(p0) + (__float_as_int(r0) << 23)),
               __int_as_float(__float_as_int(p1) + (__float_as_int(r1) << 23)));
}

// P = exp2(s a + nk) for 32 scores of one row (one hand-off part), packed for the P V MMA -- PF 0 / 1: f16 / bf16 pairs (16 words),
// PF 2: e4m3 quads (8 words; element k of the row in byte k & 3 of word k >> 2: tools/f8_probe.cu), PF 3: f16 pairs of P_hi = f16(P)
// (words 0-15) and of P_lo = f16(P - P_hi) (words 16-31), together 22 significant bits of P; the fp32 row sum accumulates
// in a packed register.  NP of every 8 element pairs take the polynomial (compile-time pattern, so the loop body is branch-free).
template <int PF, int NP>
__device__ __forceinline__ void exp_part(const float* s, f32x2 a2, f32x2 nk2, uint32_t* pk, f32x2& acc_a, f32x2& acc_b) {
  static_assert(NP == 0 || NP == 3, "exp2 mixes: all MUFU, or pairs 1, 4, 6 of every 8 on the polynomial");
  constexpr int kSel = NP == 3 ? 0x52 : 0x00;
  uint32_t half16[PF == 2 ? 16 : 1];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const f32x2 x = fma2(pack2(s[2 * i], s[2 * i + 1]), a2, nk2);
    f32x2 pp;
    float p0, p1;
    if ((kSel >> (i & 7)) & 1) {
      pp = exp2_poly2(x);
    } else {
      float x0, x1;
      unpack2(x, x0, x1);
      pp = pack2(ex2(x0), ex2(x1));
    }
    if (i & 1) acc_b = add2(acc_b, pp); else acc_a = add2(acc_a, pp);
    unpack2(pp, p0, p1);
    if constexpr (PF == 2) half16[i] = pack_e4m3(p0, p1);
    else if constexpr (PF == 3) {
      const uint32_t h = pack_f16(p0, p1);
      const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&h));
      pk[i] = h;
      pk[16 + i] = pack_f16(p0 - hf.x, p1 - hf.y);
    }
    else pk[i] = PF == 1 ? pack_bf16(p0, p1) : pack_f16(p0, p1);
  }
  if constexpr (PF == 2) {
#pragma unroll
    for (int i = 0; i < 8; ++i) pk[i] = half16[2 * i] | (half16[2 * i + 1] << 16);
  }
}

// The whole exp2 phase of one KV step: four 32-key parts, each stored to TMEM and published to the MMA warp one part
// of arithmetic later (so tcgen05.wait::st never stalls on the store just issued).  One straight-line block: ptxas
// interleaves the MUFU and polynomial work of neighbouring parts.  Sums of the two 64-key halves are kept apart
// (int8 mode folds the V block scale of each half into its exponent).
template <int PF, int NP>
__device__ __forceinline__ void exp_phase(const float* s, float a0, float a1, float nk0, float nk1, uint32_t tS,
                                          uint32_t bar0, int lane, float& sum_lo, float& sum_hi) {
  constexpr int kW = PF == 2 ? 8 : 16;             // TMEM columns of one part
  f32x2 acc[2][2] = {{pack2(0.f, 0.f), pack2(0.f, 0.f)}, {pack2(0.f, 0.f), pack2(0.f, 0.f)}};
  uint32_t pk[kParts][PF == 3 ? 32 : kW];
#pragma unroll
  for (int part = 0; part < kParts; ++part) {
    const bool hi = part >= kParts / 2;
    const float ah = hi ? a1 : a0, nk = hi ? nk1 : nk0;
    exp_part<PF, NP>(s + 32 * part, pack2(ah, ah), pack2(nk, nk), pk[part], acc[hi ? 1 : 0][0], acc[hi ? 1 : 0][1]);
    if (part > 0) {            // part-1's store was issued a whole part of arithmetic ago: publish it
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar0 + 8 * (part - 1));
    }
    if constexpr (PF == 2) tmem_st_x8(tS + kW * part, pk[part]);
    else tmem_st_x16(tS + kW * part, pk[part]);
    if constexpr (PF == 3) tmem_st_x16(tS + 64 + kW * part, pk[part] + 16);      // P_lo: columns [64, 128) of the S region
  }
  tmem_wait_st();
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive(bar0 + 8 * (kParts - 1));
  float x0, x1;
  unpack2(add2(acc[0][0], acc[0][1]), x0, x1); sum_lo = x0 + x1;
  unpack2(add2(acc[1][0], acc[1][1]), x0, x1); sum_hi = x0 + x1;
}

// Additive 16-bit mask terms of two neighbouring keys (one 32-bit word) onto their scores, in natural-log units:
//   s <- s * cn + m,   cn = softmax scale (the exponent's multiplier becomes log2 e for the rest of the step)
// one packed FMA per pair plus the two ALU ops that widen the terms (the first version spent 3 instructions per element on
// fmaf(s, a, fmaf(m, log2 e, 0)) and a per-element format select; the softmax warps' issue slots are what bounds this kernel)
template <bool BF>
__device__ __forceinline__ void add_mask_pair(float& s0, float& s1, uint32_t w, f32x2 cn2) {
  float lo, hi;
  if constexpr (BF) {
    lo = __uint_as_float(w << 16);
    hi = __uint_as_float(w & 0xffff0000u);
  } else {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w));
    lo = f.x; hi = f.y;
  }
  unpack2(fma2(pack2(s0, s1), cn2, pack2(lo, hi)), s0, s1);
}

// Cfg::kPoly of every 8 element pairs go through exp2_poly2 instead of MUFU.EX2 (on masked tiles too: the polynomial
// returns an exact zero for hidden elements, see its clamp).
// MASKED: an external mask (bool or additive, SURVEY A4 with the PyTorch placement softmax(scale * QK^T + mask)) is read by
// the softmax warps straight from global memory -- each thread owns one row, so it reads the 128 mask values of its row
// and tile with 32-byte (one sector) loads; no dense fp32 expansion pass like the reference's mfa_prepare_mask (MFABridge.swift:153-243).
template <int D, int MODE, int MASKED>      // MASKED: 0 none, 1 read in place, 2 staged by TMA
__global__ void __launch_bounds__(kThreads, 1) fwd_tc_kernel(const __grid_constant__ FwdTcParams p) {
  using C = Cfg<D, MODE, MASKED>;
  constexpr bool I8 = C::kI8, F8 = C::kF8, SPLIT = C::kSplit, I4 = C::kI4, WIDE = C::kWide, MT = C::kMaskTma;
  constexpr int PF = SPLIT ? 3 : F8 ? 2 : ((MODE == kFwdF16 || MODE == kFwdWideF16) ? 0 : 1);  // format of P (and of V): f16 / bf16 / e4m3 / f16 (hi, lo) pairs
  // e4m3 P: the exponent carries +kShift so that P' = 2^kShift P uses the format's range (max 448), and the running max
  // may lag the true one by kThr = 2 only (P' <= 2^8); 16-bit P: lag 2^8 (bf16 / fp32-range exponent, f16 P <= 256 < 65504)
  constexpr float kShift = F8 ? 6.f : 0.f;
  constexpr float kThr = F8 ? 2.f : kRescaleThreshold;
  constexpr int QT = C::kQTile, HT = C::kHalf, VT = C::kVTile, STG = C::kStage, NS = C::kStages, CHB = C::kChunkBytes;
  constexpr int SPS = C::kSPS;
  constexpr int kWg2Regs = 40;      // 8 x 232 + 4 x 40 = 504 x 32 per lane slot: an exact fit (4 x 48) leaves setmaxnreg.inc waiting forever
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  const uint32_t sQ = base, sKV = base + 2 * QT, sBar = sKV + NS * STG;
  auto q_full = [&](int t) { return sBar + 8 * t; };
  auto s_full = [&](int t) { return sBar + 16 + 8 * t; };
  auto o_full = [&](int t) { return sBar + 32 + 8 * t; };
  auto p_part = [&](int t, int k) { return sBar + 48 + 8 * (t * kParts + k); };
  auto kv_full = [&](int s) { return sBar + 112 + 8 * s; };
  auto kv_empty = [&](int s) { return sBar + 112 + 8 * NS + 8 * s; };
  const uint32_t tmem_slot = sBar + 112 + 16 * NS;
  auto o_empty = [&](int t) { return sBar + 112 + 16 * NS + 16 + 8 * t; };   // softmax warps: O_t left TMEM (fp32 split flush)
  // int4 operands: raw_full / raw_empty of the packed K ring, qraw_full / qraw_empty of the packed Q tile
  constexpr int NR = C::kRawStages, RAW = C::kRawTile;
  auto raw_full = [&](int s) { return sBar + 112 + 16 * NS + 32 + 8 * s; };
  auto raw_empty = [&](int s) { return sBar + 112 + 16 * NS + 56 + 8 * s; };
  const uint32_t qraw_full = sBar + 112 + 16 * NS + 80, qraw_empty = sBar + 112 + 16 * NS + 88;
  const uint32_t sRawK = (sBar + C::kBarBytes + 127u) & ~127u, sRawQ = sRawK + NR * RAW, sQsum = sRawQ + RAW;
  // staged external mask (MT): one 128 x 128 tile per query tile, 128-byte swizzled like the operand tiles
  auto mk_full = [&](int t) { return sBar + 112 + 16 * NS + 96 + 8 * t; };
  auto mk_empty = [&](int t) { return sBar + 112 + 16 * NS + 112 + 8 * t; };
  const uint32_t sMask = (sBar + C::kBarBytes + 1023u) & ~1023u;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp-uniform for ptxas
  // packed variable-length sequences (common.h): unmasked instantiations only -- segments do not combine with external masks
  const int* const seg_q = MASKED ? nullptr : p.cu_q;
  const int* const seg_k = MASKED ? nullptr : p.cu_k;
  // decode over a K/V cache (FwdTcParams::kv_len): the 16-bit unmasked instantiations serve it
  constexpr bool KVC = (MODE == kFwdF16 || MODE == kFwdBF16) && MASKED == 0;
  // packed query-item slots: the sequence that owns this CTA's slot, found once (the int4 barrier words, unused by KVC modes)
  int* const kv_owner = reinterpret_cast<int*>(smem_raw + (raw_full(0) - raw));
  // One CTA per work item = (batch, head, 256-row query block), x fastest so the CTAs of one head run together (K/V stay in L2).
  // KVC: q0 = first query row of sequence b in the packed Q (kv_cu_q) or 0, sq = its number of new tokens
  struct Item { int r0, h, b, hk, nt, j_lo, n, lid, half, L, q0, sq; };
  auto decode = [&](int w) {
    Item it;
    if constexpr (KVC) {
      if (p.kv_len) {        // (query item, split, KV head, sequence), query items fastest: they read the same keys
        it.half = 0; it.lid = 0;
        int qi, split;
        if (p.kv_slots) {    // packed slots: (slot, split, KV head)
          const int slot = w % p.kv_slots;
          w /= p.kv_slots;
          split = w % p.kv_nsplit;
          it.hk = w / p.kv_nsplit;
          it.b = *kv_owner;
          qi = slot - kvc_first_slot(p.kv_cu_q, it.b, p.kv_total, 2 * p.kv_sqb);
        } else {
          qi = w % p.kv_nqi;
          w /= p.kv_nqi;
          split = w % p.kv_nsplit;
          w /= p.kv_nsplit;
          it.hk = w % p.Hkv; it.b = w / p.Hkv;
        }
        it.h = it.hk * p.kv_g;
        it.q0 = p.kv_cu_q ? seg_offset(p.kv_cu_q, it.b, p.kv_total) : 0;
        it.sq = p.kv_cu_q ? kvc_seq_len(p.kv_cu_q, it.b, p.kv_total, p.Sq) : p.Sq;
        it.r0 = 2 * qi * p.kv_sqb;                                         // first token of the item
        it.nt = it.r0 + p.kv_sqb < it.sq ? 2 : 1;
        if (qi < 0 || it.r0 >= it.sq) { it.nt = 0; it.n = 0; return it; } // a slot past its sequence's rows
        it.L = kvc_len(p.kv_len, it.b, p.kv_cap);
        int klo, khi, t0, t1;
        kvc_block_key_range(p.causal, p.window, it.L, it.sq, it.r0, min(it.r0 + it.nt * p.kv_sqb, it.sq), klo, khi);
        kvc_split_tiles((p.kv_cap + 127) >> 7, p.kv_nsplit, split, t0, t1);
        it.j_lo = max(klo >> 7, t0);
        it.n = khi > klo ? max(0, min((khi + 127) >> 7, t1) - it.j_lo) : 0;
        return it;
      }
    }
    const int nqb = (p.Sq + 255) / 256;
    it.half = 0;
    if constexpr (WIDE) { it.half = w & 1; w >>= 1; }           // the two O halves of a query block run next to each other
    const int x = w % nqb, hb = w / nqb;
    const int qblk = p.causal ? nqb - 1 - x : x;                                     // heavy blocks first
    it.h = hb % p.H; it.b = hb / p.H;
    it.hk = it.h / (p.H / p.Hkv);
    it.r0 = qblk * 256;
    it.nt = (it.r0 + 128 < p.Sq) ? 2 : 1;
    int klo, khi;
    block_key_range(p.causal, p.window, p.Sq, p.Skv, seg_q, seg_k, p.nseq, it.r0, min(it.r0 + 256, p.Sq), klo, khi);
    it.j_lo = klo >> 7;
    it.n = khi > klo ? ((khi + 127) >> 7) - it.j_lo : 0;
    it.lid = 0;
    if constexpr (MASKED) {
      if (p.mtiles) {        // the list already folds in the causal / window range
        it.lid = ((p.mask_sb ? it.b : 0) * (p.mask_sh ? p.H : 1) + (p.mask_sh ? it.h : 0)) * nqb + qblk;
        it.n = __ldg(p.mcounts + it.lid);
      }
    }
    return it;
  };
  // KV tile visited at step `it` of an item
  auto tile_of = [&](const Item& im, int it) {
    if constexpr (MASKED) { if (p.mtiles) return __ldg(p.mtiles + (size_t)im.lid * p.m_nkt + it); }
    return im.j_lo + it;
  };
  if constexpr (KVC) {
    if (p.kv_len && p.kv_slots) {
      if (threadIdx.x == 0) *kv_owner = kvc_slot_owner(p.kv_cu_q, p.nbatch, p.kv_total, 2 * p.kv_sqb, (int)blockIdx.x % p.kv_slots);
      __syncthreads();
    }
    // a query-item slot without rows: no TMA, no partial (the combine kernel never reads its slot)
    if (p.kv_len && decode(blockIdx.x).nt == 0) return;
  }

  if (threadIdx.x == 256) {
    for (int t = 0; t < 2; ++t) {
      mbar_init(q_full(t), 1); mbar_init(s_full(t), 1); mbar_init(o_full(t), 1);
      for (int k = 0; k < kParts; ++k) mbar_init(p_part(t, k), 4);
    }
    for (int s = 0; s < NS; ++s) { mbar_init(kv_full(s), 1); mbar_init(kv_empty(s), 2); }   // a lone tile releases twice
    for (int t = 0; t < 2; ++t) mbar_init(o_empty(t), 4);
    if constexpr (I4) {
      for (int r = 0; r < NR; ++r) { mbar_init(raw_full(r), 1); mbar_init(raw_empty(r), 1); }
      mbar_init(qraw_full, 1); mbar_init(qraw_empty, 1);
    }
    if constexpr (MT) {
      for (int t = 0; t < 2; ++t) { mbar_init(mk_full(t), 1); mbar_init(mk_empty(t), 4); }
    }
    fence_mbar_init();
  }
  if (warp == 9) {
    if (lane == 0) { prefetch_tmap(&p.tq); prefetch_tmap(&p.tk); prefetch_tmap(&p.tv); }
    __syncwarp();
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw)), 0);

  if (warp == 9) {
    // ------------------------------------------------------------------ TMA producer
    reg_dealloc<kWg2Regs>();
    if (lane == 0) {
      const Item im = decode(blockIdx.x);
      const int r0 = im.r0, h = im.h, b = im.b, hk = im.hk, nt = im.nt, n = im.n;
      int kvi = 0;                                      // running ring index
      int kr = 0, nqraw = 0;                            // int4: packed K / Q tiles requested so far
      // one Q / K tile (or one hi / lo half of a split tile); the caller has armed the barrier with the bytes
      auto load_half = [&](uint32_t dst, const CUtensorMap* m, uint32_t bar, int row, int head, int col0 = 0) {
#pragma unroll
        for (int c = 0; c < C::kQChunks; ++c) tma_load_4d(dst + c * CHB, m, bar, col0 + c * (I8 ? 128 : 64), row, head, b);
      };
      auto load_q = [&](int t2) {
        if constexpr (I4) {              // packed tile into the raw Q buffer; the converter warp unpacks it into sQ
          if (nqraw > 0) mbar_wait(qraw_empty, (nqraw - 1) & 1);
          mbar_arrive_expect_tx(qraw_full, RAW);
          tma_load_4d(sRawQ, &p.tq, qraw_full, 0, r0 + t2 * 128, h, b);
          ++nqraw;
          return;
        }
        if constexpr (KVC) {
          if (p.kv_len) {      // GQA-packed tile: box (64, kv_sqb, G) of the (D, Sq, G, Hkv, B) map lands as rows g * kv_sqb + s
            // (packed Q: the (D, total_q, G, Hkv, 1) map from row q0; box rows past the sequence are dead rows)
            mbar_arrive_expect_tx(q_full(t2), p.kv_qbytes);
            const int qrow = im.q0 + r0 + t2 * p.kv_sqb, qb = p.kv_cu_q ? 0 : b;
#pragma unroll
            for (int c = 0; c < C::kQChunks; ++c) tma_load_5d(sQ + t2 * QT + c * CHB, &p.tq, q_full(t2), c * 64, qrow, 0, hk, qb);
            return;
          }
        }
        mbar_arrive_expect_tx(q_full(t2), QT);
        load_half(sQ + t2 * QT, &p.tq, q_full(t2), r0 + t2 * 128, h);
        if constexpr (SPLIT) load_half(sQ + t2 * QT + HT, &p.tq2, q_full(t2), r0 + t2 * 128, h);
        if constexpr (WIDE) load_half(sQ + t2 * QT + HT, &p.tq, q_full(t2), r0 + t2 * 128, h, 128);
      };
      auto load_k = [&](const CUtensorMap* m, int row, int col0 = 0) {
        if constexpr (I4) {              // packed tile into the raw ring; its operand stage (ring index kvi) is the converter's
          const int rs = kr % NR;
          mbar_wait(raw_empty(rs), ((kr / NR) & 1) ^ 1);
          mbar_arrive_expect_tx(raw_full(rs), RAW);
          tma_load_4d(sRawK + rs * RAW, m, raw_full(rs), 0, row, hk, b);
          ++kr; ++kvi;
          return;
        }
        const int s = kvi % NS;
        mbar_wait(kv_empty(s), ((kvi / NS) & 1) ^ 1);
        mbar_arrive_expect_tx(kv_full(s), HT);
        load_half(sKV + s * STG, m, kv_full(s), row, hk, col0);
        ++kvi;
      };
      auto load_v = [&](const CUtensorMap* m, int row, int col0 = 0) {
        const int s = kvi % NS;
        mbar_wait(kv_empty(s), ((kvi / NS) & 1) ^ 1);
        mbar_arrive_expect_tx(kv_full(s), VT);
#pragma unroll
        for (int c = 0; c < C::kVChunks; ++c) tma_load_4d(sKV + s * STG + c * CHB, m, kv_full(s), col0 + c * 64, row, hk, b);
        ++kvi;
      };
      bool paged = false;
      if constexpr (KVC) paged = p.kv_pages != nullptr;
      if (paged) {
        // paged K / V cache: the pools are mapped as [num_pages, page_size, Hkv, D], and a 128-key tile arrives as 128 / kv_box boxes
        // of kv_box = gcd(page_size, 128) rows, each inside one page.  Box rows are a multiple of 16, so the boxes together leave
        // the same 128-byte-swizzled image as one 128-row box.  The page ids of the next tile are read right after this tile's loads
        // are issued, so their L2 round trip overlaps the wait for a free stage.
        const int br = p.kv_box, nb = 128 / br;
        const int* bt = p.kv_pages + (size_t)b * p.kv_npb;
        int pg[8];
        auto fetch_pages = [&](int j) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int key = j * 128 + i * br;
            pg[i] = p.kv_npages;               // past the capacity: a box wholly outside the pool, which TMA fills with zeros
            if (i < nb && key < p.kv_cap) pg[i] = min(max(__ldg(bt + key / p.kv_page), 0), p.kv_npages - 1);
          }
        };
        auto load_paged = [&](const CUtensorMap* m, uint32_t bytes, int nch, int j) {
          const int s = kvi % NS;
          mbar_wait(kv_empty(s), ((kvi / NS) & 1) ^ 1);
          mbar_arrive_expect_tx(kv_full(s), bytes);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (i < nb) {
              const int prow = (j * 128 + i * br) % p.kv_page;
              for (int c = 0; c < nch; ++c)
                tma_load_4d(sKV + s * STG + c * CHB + i * br * 128, m, kv_full(s), c * 64, prow, hk, pg[i]);
            }
          }
          ++kvi;
        };
        if (n > 0) { fetch_pages(im.j_lo); load_q(0); }
        for (int it = 0; it < n; ++it) {
          load_paged(&p.tk, HT, C::kQChunks, im.j_lo + it);
          if (it == 0 && nt == 2) load_q(1);
          load_paged(&p.tv, VT, C::kVChunks, im.j_lo + it);
          if (it + 1 < n) fetch_pages(im.j_lo + it + 1);
        }
      }
      if (!paged && n > 0) load_q(0);
      for (int it = 0; it < n && !paged; ++it) {
        const int row = (tile_of(im, it) & (kTileNoMask - 1)) * 128;
        if constexpr (SPLIT) load_k(&p.tk2, row);         // K_lo first: its stage is released after the first MMA group
        load_k(&p.tk, row);
        if constexpr (WIDE) load_k(&p.tk, row, 128);      // K_b: head dims 128 .. 255
        if (it == 0 && nt == 2) load_q(1);
        load_v(&p.tv, row, WIDE ? 128 * im.half : 0);
        if constexpr (SPLIT) load_v(&p.tv2, row);         // V_lo last: only the closing MMA group of the step reads it
      }
    }
  } else if (warp == 8 || warp == 10) {
    // ------------------------------------------------------------------ MMA issuer of tile t (whole warp, one elected lane issues)
    reg_dealloc<kWg2Regs>();
    const int t = (warp - 8) >> 1;
    constexpr uint32_t FMT = (PF == 0 || PF == 3) ? 0u : 1u;      // f16 / bf16 operands of kind::f16
    constexpr uint32_t IDESC_S = I4 ? make_idesc(2, 1, 0, 0, 0, 128, 128)        // s32 += s8 * u8: K nibbles stay unsigned (see converter)
                               : I8 ? make_idesc(2, 1, 1, 0, 0, 128, 128)        // s32 += s8 * s8, K-major A and B
                                    : make_idesc(1, FMT, FMT, 0, 0, 128, 128);
    constexpr uint32_t IDESC_O = F8 ? make_idesc(1, 0, 0, 0, 1, 128, D)          // kind::f8f6f4: f32 += e4m3 P (tmem) * e4m3 V
                                    : make_idesc(1, FMT, FMT, 0, 1, 128, D);     // f32 += P (tmem) * V, V MN-major
    const uint32_t q_lo = desc_lo(sQ, 16) + t * (QT >> 4), k_lo = desc_lo(sKV, 16), v_lo = desc_lo(sKV, CHB);
    const uint32_t tS = tmem + t * 128, tO = tmem + 256 + t * D;
    // S of one KV step.  idx = ring index of the step's first stage.  Split operands: S = Q_hi K_lo^T + Q_hi K_hi^T + Q_lo K_hi^T
    // (the dropped Q_lo K_lo^T is 2^-22 of the product); the K_lo stage goes back to the producer after the first group.
    auto wait_full = [&](int idx) { mbar_wait(kv_full(idx % NS), (idx / NS) & 1); };
    auto issue_qk = [&](uint32_t a0, int idx, bool acc0) {
      const uint32_t b0 = k_lo + (idx % NS) * (STG >> 4);
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk) {
        const uint32_t off = ((kk >> 2) * CHB + (kk & 3) * 32) >> 4;
        mma_f16_ss_u(tS, a0 + off, kDescHiSw128, b0 + off, kDescHiSw128, IDESC_S, acc0 || kk > 0);
      }
    };
    auto issue_s = [&](int idx) {
      const uint32_t b0 = k_lo + (idx % NS) * (STG >> 4);
      if constexpr (I8) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)           // 32 int8 per MMA = 32 bytes of the 128-byte row
          mma_i8_ss_u(tS, q_lo + kk * 2, kDescHiSw128, b0 + kk * 2, kDescHiSw128, IDESC_S, kk > 0);
      } else {
        issue_qk(q_lo, idx, false);
      }
    };
    auto issue_o_part = [&](int idx, int part, bool acc) {
      const uint32_t b0 = v_lo + (idx % NS) * (STG >> 4);
      if constexpr (F8) {        // one K = 32 MMA per part: 8 TMEM columns of e4m3 quads, 32 key rows of 128 bytes
        mma_f8_ts_u(tO, tS + part * 8, b0 + part * (4096 >> 4), kDescHiSw128, IDESC_O, (acc || part > 0) ? 1u : 0u);
      } else {
#pragma unroll
        for (int kk = 2 * part; kk < 2 * part + 2; ++kk) {
          mma_f16_ts_u(tO, tS + kk * 8, b0 + kk * (2048 >> 4), kDescHiSw128, IDESC_O, (acc || kk > 0) ? 1u : 0u);
          if constexpr (SPLIT) mma_f16_ts_u(tO, tS + 64 + kk * 8, b0 + kk * (2048 >> 4), kDescHiSw128, IDESC_O, 1u);   // P_lo V_hi
        }
      }
    };
    int pc = 0;                                    // KV steps done by this tile
    int oe = 0;                                    // o_empty phases consumed: one per O hand-over (flush)
    const int F = SPLIT ? p.flush_steps : 0;       // fp32 split mode: O leaves TMEM every F steps (see the softmax warps)
    const Item im = decode(blockIdx.x);
    const int nt = im.nt, n = im.n;
    if (n > 0 && t < nt) {
      // a lone tile (ragged last query block) releases every ring stage for the absent one as well
      auto release = [&](int idx) { tc_commit_u(kv_empty(idx % NS)); if (nt == 1) tc_commit_u(kv_empty(idx % NS)); };
      // all of S of the step whose stages start at ring index idx: wait for the K stages, issue, publish S, free the stages
      auto do_s = [&](int idx) {
        wait_full(idx);
        tc_fence_after();
        if constexpr (SPLIT) {
          issue_qk(q_lo, idx, false);                  // Q_hi K_lo^T
          release(idx);
          wait_full(idx + 1);
          tc_fence_after();
          issue_qk(q_lo, idx + 1, true);               // Q_hi K_hi^T
          issue_qk(q_lo + (HT >> 4), idx + 1, true);   // Q_lo K_hi^T
          tc_commit_u(s_full(t));
          release(idx + 1);
        } else if constexpr (WIDE) {
          issue_qk(q_lo, idx, false);                  // Q_a K_a^T
          release(idx);
          wait_full(idx + 1);
          tc_fence_after();
          issue_qk(q_lo + (HT >> 4), idx + 1, true);   // + Q_b K_b^T
          tc_commit_u(s_full(t));
          release(idx + 1);
        } else {
          issue_s(idx);
          tc_commit_u(s_full(t));
          release(idx);
        }
      };
      mbar_wait(q_full(t), 0);
      do_s(0);
      for (int it = 0; it < n; ++it) {
        const int vi = SPS * it + (SPS == 2 ? 1 : 2), ki = SPS * (it + 1);
        wait_full(vi);
#pragma unroll
        for (int part = 0; part < kParts; ++part) {
          mbar_wait(p_part(t, part), pc & 1);
          // the first P V of a flush period (split mode) overwrites O: the softmax warps must have read the previous contents
          // out of TMEM (flush) -- one o_empty phase per hand-over
          const bool fresh = F > 0 ? (it % F == 0) : (it == 0);
          if (part == 0 && fresh && it > 0) { mbar_wait(o_empty(t), oe & 1); ++oe; }
          tc_fence_after();
          issue_o_part(vi, part, !fresh);
        }
        release(vi);
        if constexpr (SPLIT) {                         // closing group of the step: P_hi V_lo over all 128 keys
          wait_full(vi + 1);
          tc_fence_after();
          const uint32_t b0 = v_lo + ((vi + 1) % NS) * (STG >> 4);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) mma_f16_ts_u(tO, tS + kk * 8, b0 + kk * (2048 >> 4), kDescHiSw128, IDESC_O, 1u);
          release(vi + 1);
        }
        if (it + 1 < n) do_s(ki);
        else tc_commit_u(o_full(t));
        ++pc;
      }
    }
  } else if (warp < 8) {
    // ------------------------------------------------------------------ softmax warpgroups
    reg_alloc<232>();
    const int t = warp >> 2;
    const int row = (warp & 3) * 32 + lane;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t tS = tmem + lane_base + t * 128;
    const uint32_t tO = tmem + lane_base + 256 + t * D;
    int pc = 0;                                            // KV steps done by this tile (barrier phases)
    int mkc = 0;                                           // staged mask tiles consumed by this tile
    if (t == 1) named_bar_arrive(2, 256);                  // the first turn belongs to tile 0
    const Item im = decode(blockIdx.x);
    const int r0 = im.r0, h = im.h, b = im.b, hk = im.hk, nt = im.nt, n = im.n;
    const int r = r0 + t * 128 + row;
    float m = -CUDART_INF_F, l = 0.f;                      // m in scaled log2 units (score * scale * log2 e)
    int clo, chi;                                          // visible keys of this row: [clo, chi]
    bool kvc = false;
    if constexpr (KVC) kvc = p.kv_len != nullptr;
    if (kvc) {
      // token s of query head g = row / kv_sqb; rows past G * kv_sqb (stale shared memory) and tokens past the sequence's
      // (zero-filled, or another sequence's) see no key
      const int s = r0 + t * p.kv_sqb + row % p.kv_sqb;
      clo = chi = 0;
      if (row < p.kv_rows && s < im.sq) kvc_row_key_range(p.causal, p.window, im.L, im.sq, s, clo, chi);
    } else {
      row_key_range(p.causal, p.window, p.Sq, p.Skv, seg_q, seg_k, p.nseq, r, clo, chi);
    }
    --chi;
    // int8 mode: per-row Q scale (folded with c), per-64-key K and V block scales
    float qsc = p.c;
    const float* ksp = nullptr;
    const float* vsp = nullptr;
    if constexpr (I8) {
      const int rq = min(r, p.Sq - 1);
      qsc = (p.qs ? p.qs[((size_t)b * p.H + h) * p.sq_ + rq / p.qbr] : p.qs1) * p.c;
      ksp = p.ks ? p.ks + ((size_t)b * p.Hkv + hk) * p.sk_ : nullptr;
      vsp = p.vs ? p.vs + ((size_t)b * p.Hkv + hk) * p.sv_ : nullptr;
    }
    // split mode: the operands were scaled by powers of two into fp16's range (qs / ks / vs point at the inverse scales)
    if constexpr (SPLIT) qsc = p.c * __ldg(p.qs) * __ldg(p.ks);
    float sb_row = p.s_bias;                               // offset of the widened integer score of this row (int4: set at step 0)
    float m_flush = -CUDART_INF_F;                         // split mode: running max the flushed part of O (in global memory) is scaled by
    int nflush = 0;
    const int dv_row = p.dv > 0 ? p.dv : D;                // head dims this row holds in global memory
    const bool v_blocks = I8 && !F8 && vsp != nullptr;     // (e4m3 V carries one scale per (b, head): applied in the epilogue)
    const bool pingpong = nt == 2;

    if (t < nt) {
      // int8 mode: raw K / V block scales of the two 64-key halves of a tile.  They are fetched one KV step ahead (right
      // after S of the current step has been read), so the L2 / HBM latency of these loads never sits between the
      // s_full wait and the exp2 phase (it cost ~900 clk per step when the loads were issued at the top of the step).
      float ksn0 = p.ks1, ksn1 = p.ks1, vsn0 = 1.f, vsn1 = 1.f;
      int jt_next = n > 0 ? tile_of(im, 0) : 0;        // tile index of the coming step (read one step ahead)
      auto fetch_scales = [&](int jt) {
        if constexpr (I8) {
          const int c0 = (jt & (kTileNoMask - 1)) * 128;
          if (ksp) {
            ksn0 = __ldg(ksp + min(c0 / p.kbr, p.nbk - 1));
            ksn1 = __ldg(ksp + min((c0 + 64) / p.kbr, p.nbk - 1));
          }
          if (v_blocks) {
            vsn0 = __ldg(vsp + min(c0 / p.vbr, p.nbv - 1));
            vsn1 = __ldg(vsp + min((c0 + 64) / p.vbr, p.nbv - 1));
          }
        }
      };
      if (n > 0) fetch_scales(jt_next);
      for (int it = 0; it < n; ++it) {
        const int c0 = (jt_next & (kTileNoMask - 1)) * 128;
        const bool mask_noop = (jt_next & kTileNoMask) != 0;
        // multipliers of the two 64-key halves of this tile (int8: blocks are multiples of 64 keys)
        float a0 = qsc, a1 = qsc, lv0 = 0.f, lv1 = 0.f, iv0 = 1.f, iv1 = 1.f;
        float cb0 = 0.f, cb1 = 0.f;              // int8: - (s_bias [+ 8 rowsum(q)]) a_h, folded into every addend that follows a multiplication by a_h
        if constexpr (I8) {
          a0 = qsc * ksn0;
          a1 = qsc * ksn1;
          cb0 = -sb_row * a0;
          cb1 = -sb_row * a1;
          if (v_blocks) {
            lv0 = log2f(vsn0); lv1 = log2f(vsn1);    // bf16 P' = P v_h has fp32's exponent range: no reference scale needed
            iv0 = 1.f / vsn0; iv1 = 1.f / vsn1;
          }
        }
        mbar_wait(s_full(t), pc & 1);
        ++pc;
        tc_fence_after();
        if constexpr (SPLIT) {
          // fp32 split mode, every flush_steps steps: O leaves TMEM for an fp32 scratch tile in global memory,
          //   O_flushed = O_flushed 2^(m_flush - m) + O_tmem,
          // and the next P V starts a fresh accumulator.  tcgen05.mma adds into TMEM with truncation (~2^-24 of the accumulator per
          // MMA, 24 MMAs per step): bounded accumulator lifetimes keep that bias at ~7e-6 of O; the sums across periods are
          // round-to-nearest FMAs in registers.  S of this step being ready means the P V of the step before has retired.
          if (p.flush_steps > 0 && it > 0 && it % p.flush_steps == 0) {
            const float fs = (nflush > 0 && m_flush != -CUDART_INF_F) ? ex2(m_flush - m) : 0.f;
            // the flushed part lives in a scratch tile private to this (item, tile), laid out [column / 4][row][4]: the 32 rows
            // of a warp touch consecutive 16-byte units, so every access is a fully coalesced 512-byte request (row-major rows
            // of the output would cost 32 sectors in 32 lines per request)
            float4* fbuf = reinterpret_cast<float4*>(p.flush_buf) + ((size_t)blockIdx.x * 2 + t) * (size_t)(D / 4) * 128 + row;
#pragma unroll
            for (int ch = 0; ch < D / 32; ++ch) {
              uint32_t ou[32];
              tmem_ld_x32(tO + ch * 32, ou);
              tmem_wait_ld();
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float4* dst = fbuf + (size_t)(ch * 8 + i) * 128;
                float4 o4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (nflush > 0) o4 = *dst;
                *dst = make_float4(fmaf(o4.x, fs, __uint_as_float(ou[4 * i])), fmaf(o4.y, fs, __uint_as_float(ou[4 * i + 1])),
                                   fmaf(o4.z, fs, __uint_as_float(ou[4 * i + 2])), fmaf(o4.w, fs, __uint_as_float(ou[4 * i + 3])));
              }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(o_empty(t));
            m_flush = m;
            ++nflush;
          }
        }
        if constexpr (I4) {
          // unsigned K nibbles: S_true = S_mma - 8 sum_d q[row][d]; the row constant joins the widening offset (both exact integers
          // in fp32).  The converter wrote the sums before it published Q, S of this item was computed from that Q.
          if (it == 0) {
            sb_row = p.s_bias + 8.f * (float)(int)ld_shared_u32(sQsum + t * 512 + row * 4);
            cb0 = -sb_row * a0;
            cb1 = -sb_row * a1;
          }
        }
        uint32_t su[128];
        tmem_ld_x32(tS, su);
        tmem_ld_x32(tS + 32, su + 32);
        tmem_ld_x32(tS + 64, su + 64);
        tmem_ld_x32(tS + 96, su + 96);
        tmem_wait_ld();
        float* s = reinterpret_cast<float*>(su);
        if (it + 1 < n) { jt_next = tile_of(im, it + 1); fetch_scales(jt_next); }
        if constexpr (I8) {
          // Widening without a conversion instruction: (s << k) plus the bit pattern of B = 1.5 * 2^(23-k), read as a float, IS
          // B + s (exact for |s| <= 2^(22-k)), and the - B a_h that undoes the offset rides in the addend of the multiply-add
          // that scales the score anyway (cb_h above).  One integer multiply-add per score on the FMA / ALU pipes instead of I2FP
          // on the XU pipe, which the exp2 MUFUs need (16 / clk / SM: 1157 clk per tile and step in round 1,
          // profiles/r01d_int8_notes.txt).  k is the largest shift the code range allows (int8: |s| <= 2^21, k = 1; int4:
          // |s| <= 2^13, k = 8): the addend nk_h = cb_h + ... is ONE fp32, so its rounding, <= 2^-25 B a_h, is the error of the
          // scaled score -- 0.19 a_h (int8) / 1.5e-3 a_h (int4, whose a_h is ~300x larger), far below one quantum a_h of S.
          const int smul = p.s_mul;
          const uint32_t sadd = p.s_add;
#pragma unroll
          for (int i = 0; i < 128; ++i) su[i] = su[i] * smul + sadd;
        }
        if (MT && !mask_noop) {
          if constexpr (MT) {
            // the mask tile of this (step, query tile) is in shared memory (TMA, 128-byte swizzle: 16-byte unit j of row r sits
            // at j ^ (r & 7), so the eight rows of a quarter warp read eight different units -- no bank conflicts); rows / keys
            // past the tensor's extent arrive as zeros (bool: hidden; additive: + 0, the range rule below hides them)
            mbar_wait(mk_full(t), mkc & 1);
            ++mkc;
            const uint32_t mrow = sMask + (uint32_t)t * C::kMaskTile + (uint32_t)row * 128u;
            const uint32_t sw = (uint32_t)(row & 7);
            if (p.mask_kind == kMaskBool) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {                         // 16 keys per unit
                float f0, f1, f2, f3;
                ld_shared_v4(mrow + (((uint32_t)j ^ sw) << 4), f0, f1, f2, f3);
                const uint32_t w4[4] = {__float_as_uint(f0), __float_as_uint(f1), __float_as_uint(f2), __float_as_uint(f3)};
#pragma unroll
                for (int k = 0; k < 16; ++k)
                  if (((w4[k >> 2] >> (8 * (k & 3))) & 0xffu) == 0) s[16 * j + k] = -CUDART_INF_F;
              }
            } else {
              // (staged masks exist for the 16-bit operand modes only: a0 == a1 == scale * log2 e, no integer offsets)
              const float cn = a0 * kLn2;
              const f32x2 cn2 = pack2(cn, cn);
              auto apply = [&](auto is_bf) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {                       // 64-key half = one 16 KB chunk
#pragma unroll
                  for (int j = 0; j < 8; ++j) {                     // 8 keys per unit
                    float f0, f1, f2, f3;
                    ld_shared_v4(mrow + (uint32_t)g * 16384u + (((uint32_t)j ^ sw) << 4), f0, f1, f2, f3);
                    const uint32_t w4[4] = {__float_as_uint(f0), __float_as_uint(f1), __float_as_uint(f2), __float_as_uint(f3)};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                      const int i = 64 * g + 8 * j + 2 * k;
                      add_mask_pair<decltype(is_bf)::value>(s[i], s[i + 1], w4[k], cn2);
                    }
                  }
                }
              };
              if (p.mask_scalar == kMaskBF16) apply(std::true_type{}); else apply(std::false_type{});
              a0 = a1 = kLog2e;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(mk_empty(t));                // the producer may refill this tile's buffer
          }
        } else if (!MT && MASKED && !mask_noop) {
          const int rq = min(r, p.Sq - 1);
          const long long eoff = (long long)b * p.mask_sb + (long long)h * p.mask_sh + (long long)rq * p.mask_sq + c0;
          const int ncol = min(128, p.Skv - c0);
          if (p.mask_kind == kMaskBool) {
            const uint8_t* mp = reinterpret_cast<const uint8_t*>(p.mask) + eoff;
            if (ncol == 128 && (reinterpret_cast<uintptr_t>(mp) & 31) == 0) {
#pragma unroll
              for (int c = 0; c < 4; ++c) {                       // 32 bytes = one sector per request
                uint32_t w[8];
                ldg256(mp + 32 * c, w);
#pragma unroll
                for (int k = 0; k < 32; ++k)
                  if (((w[k >> 2] >> (8 * (k & 3))) & 0xffu) == 0) s[32 * c + k] = -CUDART_INF_F;
              }
            } else {
#pragma unroll
              for (int i = 0; i < 128; ++i)
                if (i < ncol && __ldg(mp + i) == 0) s[i] = -CUDART_INF_F;
            }
          } else {
            // additive: fold the scale now (s <- s a_h + mask log2 e), the multipliers become 1 for the rest of the step
            bool mask_folded = false;
            if (p.mask_scalar == kMaskF32) {
              const float* mp = reinterpret_cast<const float*>(p.mask) + eoff;
              if (!I8 && ncol == 128 && (reinterpret_cast<uintptr_t>(mp) & 31) == 0) {
                const float cn = a0 * kLn2;                       // s <- s * scale + m, one FMA per element (see add_mask_pair)
#pragma unroll
                for (int c = 0; c < 16; ++c) {                    // 32 bytes = one sector per request
                  uint32_t w[8];
                  ldg256(mp + 8 * c, w);
#pragma unroll
                  for (int k = 0; k < 8; ++k) s[8 * c + k] = fmaf(s[8 * c + k], cn, __uint_as_float(w[k]));
                }
                a0 = a1 = kLog2e;
                cb0 = cb1 = 0.f;
                mask_folded = true;
              } else if (ncol == 128 && (reinterpret_cast<uintptr_t>(mp) & 31) == 0) {
#pragma unroll
                for (int c = 0; c < 16; ++c) {                    // 32 bytes = one sector per request
                  uint32_t w[8];
                  ldg256(mp + 8 * c, w);
                  const float ah = c < 8 ? a0 : a1;
#pragma unroll
                  for (int k = 0; k < 8; ++k) s[8 * c + k] = fmaf(s[8 * c + k], ah, fmaf(__uint_as_float(w[k]), kLog2e, c < 8 ? cb0 : cb1));
                }
              } else {
#pragma unroll
                for (int i = 0; i < 128; ++i)
                  s[i] = fmaf(s[i], i < 64 ? a0 : a1, fmaf(i < ncol ? __ldg(mp + i) : 0.f, kLog2e, i < 64 ? cb0 : cb1));
              }
            } else {
              const uint16_t* mp = reinterpret_cast<const uint16_t*>(p.mask) + eoff;
              const bool bf = p.mask_scalar == kMaskBF16;
              auto widen = [&](uint32_t bits) {
                return bf ? __uint_as_float(bits << 16) : __half2float(__ushort_as_half((unsigned short)bits));
              };
              if (!I8 && ncol == 128 && (reinterpret_cast<uintptr_t>(mp) & 31) == 0) {
                // same arithmetic as the staged route (bit-identical results): s <- s * scale + m in natural-log units
                const float cn = a0 * kLn2;
                const f32x2 cn2 = pack2(cn, cn);
                auto apply = [&](auto is_bf) {
#pragma unroll
                  for (int g = 0; g < 2; ++g) {                   // 4 requests of 32 bytes in flight, then their 64 terms
                    uint32_t w[4][8];
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4) ldg256(mp + 16 * (4 * g + k4), w[k4]);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4) {
                      const int c = 4 * g + k4;
#pragma unroll
                      for (int k = 0; k < 8; ++k) add_mask_pair<decltype(is_bf)::value>(s[16 * c + 2 * k], s[16 * c + 2 * k + 1], w[k4][k], cn2);
                    }
                  }
                };
                if (bf) apply(std::true_type{}); else apply(std::false_type{});
                a0 = a1 = kLog2e;
                cb0 = cb1 = 0.f;
                mask_folded = true;
              } else if (ncol == 128 && (reinterpret_cast<uintptr_t>(mp) & 31) == 0) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {                     // 4 requests of 32 bytes in flight, then their 64 terms
                  uint32_t w[4][8];
#pragma unroll
                  for (int k4 = 0; k4 < 4; ++k4) ldg256(mp + 16 * (4 * g + k4), w[k4]);
                  const float ah = g == 0 ? a0 : a1, cbh = g == 0 ? cb0 : cb1;
#pragma unroll
                  for (int k4 = 0; k4 < 4; ++k4) {
                    const int c = 4 * g + k4;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                      s[16 * c + 2 * k] = fmaf(s[16 * c + 2 * k], ah, fmaf(widen(w[k4][k] & 0xffffu), kLog2e, cbh));
                      s[16 * c + 2 * k + 1] = fmaf(s[16 * c + 2 * k + 1], ah, fmaf(widen(w[k4][k] >> 16), kLog2e, cbh));
                    }
                  }
                }
              } else {
#pragma unroll
                for (int i = 0; i < 128; ++i)
                  s[i] = fmaf(s[i], i < 64 ? a0 : a1, fmaf(i < ncol ? widen(__ldg(mp + i)) : 0.f, kLog2e, i < 64 ? cb0 : cb1));
              }
            }
            if (!mask_folded) {
              a0 = a1 = 1.f;
              cb0 = cb1 = 0.f;
            }
          }
        }
        const bool need_mask = (c0 < clo) || (c0 + 127 > chi);
        const bool any_mask = __any_sync(0xffffffffu, need_mask);
        if (any_mask) {
          const int lo_i = clo - c0, hi_i = chi - c0;
#pragma unroll
          for (int i = 0; i < 128; ++i) s[i] = (i < lo_i || i > hi_i) ? -CUDART_INF_F : s[i];
        }
        float mxa = s[0], mxb = s[1], mxc = s[64], mxd = s[65];
#pragma unroll
        for (int i = 2; i < 64; i += 2) {
          mxa = fmaxf(mxa, s[i]); mxb = fmaxf(mxb, s[i + 1]); mxc = fmaxf(mxc, s[64 + i]); mxd = fmaxf(mxd, s[65 + i]);
        }
        // per-half maxima to scaled log2 units; a_h > 0 so the max commutes with the scaling (-inf if all masked)
        float mx;
        if constexpr (I8) mx = fmaxf(fmaf(fmaxf(mxa, mxb), a0, cb0), fmaf(fmaxf(mxc, mxd), a1, cb1));
        else mx = fmaxf(fmaxf(mxa, mxb), fmaxf(mxc, mxd)) * a0;
        float m_new = fmaxf(m, mx);
        const bool grow = (m_new - m) > kThr;                       // false when both are -inf (NaN compare)
        if (!grow) m_new = m;
        if (__any_sync(0xffffffffu, grow)) {
          const float alpha = grow ? ex2(m - m_new) : 1.f;          // m = -inf -> 0
          l *= alpha;
          if (it > 0) {
#pragma unroll
            for (int ch = 0; ch < D / 16; ++ch) {           // 16 columns at a time: the 128 scores stay live in registers
              uint32_t ou[16];
              tmem_ld_x16(tO + ch * 16, ou);
              tmem_wait_ld();
#pragma unroll
              for (int i = 0; i < 16; ++i) ou[i] = __float_as_uint(__uint_as_float(ou[i]) * alpha);
              tmem_st_x16(tO + ch * 16, ou);
            }
          }
        }
        m = m_new;
        const float mm = (m == -CUDART_INF_F) ? 0.f : m;
        // int8 mode: the V scale of each 64-key half rides in the exponent (P' = P v_h feeds the P V MMA; l takes
        // sum(P') / v_h), so the inner loop is the same as the 16-bit one.
        const float nk0 = (lv0 - mm) + (cb0 + kShift), nk1 = (lv1 - mm) + (cb1 + kShift);
        float sum_lo, sum_hi;
        // exp2 turn-taking: the two tiles' exp2 phases are MUFU-bound and share the four SMSPs, so run them one after
        // the other (tile 0 first) -- this locks the tiles in anti-phase: one is in exp2 while the tensor pipe works
        // for the other.  Left alone they drift in phase (the in-order tensor pipe queues S_1 right behind S_0) and
        // each exp2 phase takes twice as long (profiles/: timeline).  Strict alternation: tile 0 takes its k-th turn on the
        // credit tile 1 posts after its (k-1)-th (the first credit is posted before the KV loop), so neither named barrier ever
        // sees two arrivals of one side in a row.  (A turn taken without the credit lets tile 0 arrive twice on barrier 3, and
        // the barrier then completes without tile 1 -- profiles/r02/r02e_watchdog_pingpong.txt.)
        if (pingpong) {
          if (t == 0) named_bar_sync(2, 256);
          else named_bar_sync(3, 256);
        }
        exp_phase<PF, C::kPoly>(s, a0, a1, nk0, nk1, tS, p_part(t, 0), lane, sum_lo, sum_hi);
        if (pingpong) {
          if (t == 0) named_bar_arrive(3, 256);
          else named_bar_arrive(2, 256);
        }
        l += sum_lo * iv0 + sum_hi * iv1;
      }
      // ---------------------------------------------------------------- epilogue: O / l, L = m + log2(l)
      if (n > 0) {
        mbar_wait(o_full(t), 0);
        tc_fence_after();
      }
      float inv = (l > 0.f ? 1.f / l : 0.f) * ((I8 && !v_blocks) ? p.vs1 : 1.f);
      if constexpr (F8) { if (p.vs) inv = (l > 0.f ? 1.f / l : 0.f) * __ldg(p.vs + (size_t)b * p.Hkv + hk); }     // per-(b, head) scale of the e4m3 V
      if constexpr (SPLIT) inv *= __ldg(p.vs);
      const bool live = kvc ? row < p.kv_rows : r < p.Sq;
      // zero-padded head dims: the columns past the true head dim p.dv are not written
      const bool padded_d = p.dv > 0 && p.dv < (WIDE ? 256 : D);
      const int dv_tile = p.dv - (WIDE ? 128 * im.half : 0);
      const size_t orow = (size_t)b * p.o_sb + (size_t)h * p.o_sh + (size_t)r * p.o_ss + (WIDE ? 128 * im.half : 0);   // wide: this CTA's half of O
      const size_t lrow = kvc ? ((size_t)blockIdx.x * 2 + t) * p.kv_rows + row : ((size_t)b * p.H + h) * p.lse_sh + r;
      float l_out = l > 0.f ? m + log2f(l) - kShift : -CUDART_INF_F;
      // accumulate mode (ring attention): the partial of this launch is merged in place with the (O, L) already there,
      //   L = log2(2^L_old + 2^L_new),  O = O_old 2^(L_old - L) + O_new 2^(L_new - L)      (fp32 O only)
      float c_old = 0.f;
      const bool acc_mode = p.accumulate && p.o_dtype == kF32;
      const bool tma_out = p.o_tma && !acc_mode;
      if (tma_out) {
        // the staging area reuses the operand memory: wait until the other tile has retired its last MMA too
        if (n > 0 && nt == 2) { mbar_wait(o_full(t ^ 1), 0); tc_fence_after(); }
      }
      if (acc_mode && live) {
        const float l_old = p.lse[lrow];
        const float mx = fmaxf(l_old, l_out);
        if (mx != -CUDART_INF_F) {
          const float w_old = exp2f(l_old - mx), w_new = exp2f(l_out - mx);     // exp2(-inf) = 0
          const float tot = w_old + w_new;
          c_old = w_old / tot;
          inv *= w_new / tot;
          l_out = mx + log2f(tot);
        }
      }
#pragma unroll
      uint32_t oall[D];
      if (n > 0) {
#pragma unroll
        for (int ch = 0; ch < D / 32; ++ch) tmem_ld_x32(tO + ch * 32, oall + ch * 32);
        tmem_wait_ld();
        if constexpr (SPLIT) {
          if (nflush > 0) {        // + what the flushes left in the scratch tile, brought to the final running max
            const float fs = m_flush != -CUDART_INF_F ? ex2(m_flush - m) : 0.f;
            const float4* src = reinterpret_cast<const float4*>(p.flush_buf) + ((size_t)blockIdx.x * 2 + t) * (size_t)(D / 4) * 128 + row;
#pragma unroll
            for (int i = 0; i < D / 4; ++i) {
              const float4 g4 = src[(size_t)i * 128];
              oall[4 * i] = __float_as_uint(fmaf(g4.x, fs, __uint_as_float(oall[4 * i])));
              oall[4 * i + 1] = __float_as_uint(fmaf(g4.y, fs, __uint_as_float(oall[4 * i + 1])));
              oall[4 * i + 2] = __float_as_uint(fmaf(g4.z, fs, __uint_as_float(oall[4 * i + 2])));
              oall[4 * i + 3] = __float_as_uint(fmaf(g4.w, fs, __uint_as_float(oall[4 * i + 3])));
            }
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < D; ++i) oall[i] = 0u;
      }
#pragma unroll
      for (int ch = 0; ch < D / 32; ++ch) {
        const uint32_t* ou = oall + ch * 32;
        if (tma_out && p.o_dtype == kF32) {
          // 32 columns of this row -> one 128-byte line of the swizzled staging chunk (16-byte unit j lands at j ^ (row & 7):
          // the layout the fp32 output tensor map expects, and conflict-free for the 32 rows of a warp)
          const uint32_t line = base + (uint32_t)(t * (D / 32) + ch) * (128u * 128u) + (uint32_t)row * 128u;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            st_shared_v4(line + (uint32_t)((i ^ (row & 7)) << 4), __uint_as_float(ou[4 * i]) * inv, __uint_as_float(ou[4 * i + 1]) * inv,
                         __uint_as_float(ou[4 * i + 2]) * inv, __uint_as_float(ou[4 * i + 3]) * inv);
        } else if (tma_out) {
          // 16-bit O: a staging chunk is 64 columns wide (128 bytes per row); these 32 columns are half a line (4 units)
          const uint32_t line = base + (uint32_t)(t * (D / 64) + (ch >> 1)) * (128u * 128u) + (uint32_t)row * 128u;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            uint32_t w[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float a = __uint_as_float(ou[8 * i + 2 * k]) * inv, bb = __uint_as_float(ou[8 * i + 2 * k + 1]) * inv;
              w[k] = p.o_dtype == kBF16 ? pack_bf16(a, bb) : pack_f16(a, bb);
            }
            const int unit = (ch & 1) * 4 + i;
            st_shared_v4(line + (uint32_t)((unit ^ (row & 7)) << 4), __uint_as_float(w[0]), __uint_as_float(w[1]),
                         __uint_as_float(w[2]), __uint_as_float(w[3]));
          }
        } else if (live && padded_d) {
          // zero-padded head dim without the TMA-store epilogue (rare: accumulate mode, views TMA cannot describe): element-wise,
          // stopping at the true head dim
          const int nv = dv_tile - ch * 32;
#pragma unroll
          for (int i = 0; i < 32; ++i) {         // fully unrolled: the registers of O must keep static indices
            if (i >= nv) continue;
            const float val = __uint_as_float(ou[i]) * inv;
            if (p.o_dtype == kF32) {
              float* dst = reinterpret_cast<float*>(p.o) + orow + ch * 32 + i;
              *dst = acc_mode ? fmaf(*dst, c_old, val) : val;
            } else {
              uint16_t* dst = reinterpret_cast<uint16_t*>(p.o) + orow + ch * 32 + i;
              *dst = (uint16_t)((p.o_dtype == kBF16 ? pack_bf16(val, 0.f) : pack_f16(val, 0.f)) & 0xffffu);
            }
          }
        } else if (live) {
          if (p.o_dtype == kF32) {
            float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.o) + orow + ch * 32);
            if (acc_mode && (reinterpret_cast<uintptr_t>(dst) & 31) == 0) {
              // read-modify-write of the running O in 32-byte (one sector) pieces: half the LSU requests of float4
              float* d8 = reinterpret_cast<float*>(dst);
              float old[32];
#pragma unroll
              for (int i = 0; i < 4; ++i) ld_global_v8(d8 + 8 * i, old + 8 * i);
#pragma unroll
              for (int i = 0; i < 32; ++i) old[i] = fmaf(old[i], c_old, __uint_as_float(ou[i]) * inv);
#pragma unroll
              for (int i = 0; i < 4; ++i) st_global_v8(d8 + 8 * i, old + 8 * i);
            } else if (acc_mode) {
              float4 old[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) old[i] = dst[i];
#pragma unroll
              for (int i = 0; i < 8; ++i)
                dst[i] = make_float4(fmaf(old[i].x, c_old, __uint_as_float(ou[4 * i]) * inv),
                                     fmaf(old[i].y, c_old, __uint_as_float(ou[4 * i + 1]) * inv),
                                     fmaf(old[i].z, c_old, __uint_as_float(ou[4 * i + 2]) * inv),
                                     fmaf(old[i].w, c_old, __uint_as_float(ou[4 * i + 3]) * inv));
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i)
                dst[i] = make_float4(__uint_as_float(ou[4 * i]) * inv, __uint_as_float(ou[4 * i + 1]) * inv,
                                     __uint_as_float(ou[4 * i + 2]) * inv, __uint_as_float(ou[4 * i + 3]) * inv);
            }
          } else {
            uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p.o) + orow + ch * 32);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              uint32_t w[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float a = __uint_as_float(ou[8 * i + 2 * k]) * inv, bb = __uint_as_float(ou[8 * i + 2 * k + 1]) * inv;
                w[k] = p.o_dtype == kBF16 ? pack_bf16(a, bb) : pack_f16(a, bb);
              }
              dst[i] = make_uint4(w[0], w[1], w[2], w[3]);
            }
          }
        }
      }
      if (tma_out) {
        fence_proxy_async_smem();
        named_bar_sync(4 + t, 128);
        if ((threadIdx.x & 127) == 0) {
          if (p.o_dtype == kF32) {
            // K/V-cache partials go to the scratch tile (tile t, item) of the [items, 2, kv_rows, D] map
            const int y = kvc ? 0 : r0 + t * 128, z = kvc ? t : h, w = kvc ? (int)blockIdx.x : b;
#pragma unroll
            for (int ch = 0; ch < D / 32; ++ch)
              tma_store_4d(&p.to, base + (uint32_t)(t * (D / 32) + ch) * (128u * 128u), ch * 32 + (WIDE ? 128 * im.half : 0), y, z, w);
          } else {
#pragma unroll
            for (int ch = 0; ch < D / 64; ++ch)
              tma_store_4d(&p.to, base + (uint32_t)(t * (D / 64) + ch) * (128u * 128u), ch * 64 + (WIDE ? 128 * im.half : 0), r0 + t * 128, h, b);
          }
          bulk_commit();
          bulk_wait_read();           // the CTA may exit (and free its shared memory) once the TMA has read the tile
        }
      }
      if (live && p.lse && (!WIDE || im.half == 0)) p.lse[lrow] = l_out;
    }
    if (t == 0) named_bar_sync(2, 256);                    // take the credit nobody will use: the barriers end balanced
  }
  else {
    reg_dealloc<kWg2Regs>();      // warp 11 (setmaxnreg is warpgroup-wide): idle, the mask producer, or the int4 converter
    if constexpr (MT) {
      // ---------------------------------------------------------------- external mask through shared memory: dense masks
      // ([., ., Sq, Skv] with 1- or 2-byte elements) come in by TMA, one 128 x 128 tile per (KV step, query tile), instead of
      // being read row by row by the softmax warps (32 lines per warp request straight to L2: the L1 tag stage, one line per
      // clock, bounded the masked forward at 2.7x the unmasked time -- profiles/r01p_bench_mask_fwd_bwd.json).  The buffer of
      // a tile is refilled as soon as its four softmax warps have applied it, a whole KV step before it is needed again.
      if (lane == 0) {
        prefetch_tmap(&p.tm);
        // the mask streams through once (up to GBs): evict-first keeps it from pushing the K / V tiles the other CTAs of a
        // head re-read out of L2
        const uint64_t pol = l2_policy_evict_first();
        const bool one_byte = p.mask_kind == kMaskBool;
        int mc[2] = {0, 0};
        const Item im = decode(blockIdx.x);
        const int mb = p.mask_sb ? im.b : 0, mh = p.mask_sh ? im.h : 0;
        for (int it = 0; it < im.n; ++it) {
          const int jt = tile_of(im, it);
          if (jt & kTileNoMask) continue;
          const int c0 = (jt & (kTileNoMask - 1)) * 128;
          for (int t = 0; t < im.nt; ++t) {
            if (mc[t] > 0) mbar_wait(mk_empty(t), (mc[t] - 1) & 1);
            const uint32_t dst = sMask + (uint32_t)t * C::kMaskTile;
            if (one_byte) {
              mbar_arrive_expect_tx(mk_full(t), 16384);
              tma_load_4d_hint(dst, &p.tm, mk_full(t), c0, im.r0 + t * 128, mh, mb, pol);
            } else {
              mbar_arrive_expect_tx(mk_full(t), 32768);
              tma_load_4d_hint(dst, &p.tm, mk_full(t), c0, im.r0 + t * 128, mh, mb, pol);
              tma_load_4d_hint(dst + 16384, &p.tm, mk_full(t), c0 + 64, im.r0 + t * 128, mh, mb, pol);
            }
            ++mc[t];
          }
        }
      }
    }
    if constexpr (I4) {
      // ---------------------------------------------------------------- int4 -> int8 in shared memory (north_star item 2;
      // the reference dequantises on load as well: MFA/GEMM/GEMMHeaders.swift:757-772).  TMA delivers the packed tile (128 rows x
      // 64 bytes, byte j = codes 2j | 2j+1 << 4, each stored + 8: GEMMQuantization.swift:501-516); this warp expands it into the
      // 128-byte-swizzled K-major operand tile the MMA reads.  Lane = one 16-byte unit (32 codes) of a row per pass, 16 passes per
      // tile: reads are consecutive, the two 16-byte stores of a pass land on 8 distinct bank groups per quarter warp.
      //   K: nibbles stay UNSIGNED (u8 operand): sum_d q (n - 8) = sum_d q n - 8 sum_d q, and the second term is a per-row constant
      //      the softmax warps fold into their addend -- so a K tile costs split + interleave only (5 ops per 8 codes);
      //   Q: signed codes (n ^ 8, sign-extended), and the row sums of the codes go to sQsum for that correction.
      auto unpack_tile = [&](uint32_t src, uint32_t dst, auto is_q, uint32_t qsum_addr) {
#pragma unroll 1
        for (int i = 0; i < 16; ++i) {
          const int id = i * 32 + lane, row = id >> 2, su = id & 3;
          float f0, f1, f2, f3;
          ld_shared_v4(src + id * 16, f0, f1, f2, f3);
          const uint32_t wv[4] = {__float_as_uint(f0), __float_as_uint(f1), __float_as_uint(f2), __float_as_uint(f3)};
          uint32_t o[8];
          int rs = 0;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            uint32_t lo = wv[k] & 0x0f0f0f0fu, hi = (wv[k] >> 4) & 0x0f0f0f0fu;
            if constexpr (decltype(is_q)::value) {
              lo ^= 0x08080808u; hi ^= 0x08080808u;                          // n - 8 as a 4-bit two's complement ...
              lo |= (lo & 0x08080808u) * 30u; hi |= (hi & 0x08080808u) * 30u; // ... sign-extended to the byte (0x08 * 30 = 0xF0)
              rs = __dp4a((int)lo, 0x01010101, rs);
              rs = __dp4a((int)hi, 0x01010101, rs);
            }
            o[2 * k] = __byte_perm(lo, hi, 0x5140);        // codes 0 1 2 3 of this word
            o[2 * k + 1] = __byte_perm(lo, hi, 0x7362);    // codes 4 5 6 7
          }
          const uint32_t line = dst + (uint32_t)row * 128u;
          st_shared_v4(line + (uint32_t)(((2 * su) ^ (row & 7)) << 4), __uint_as_float(o[0]), __uint_as_float(o[1]),
                       __uint_as_float(o[2]), __uint_as_float(o[3]));
          st_shared_v4(line + (uint32_t)(((2 * su + 1) ^ (row & 7)) << 4), __uint_as_float(o[4]), __uint_as_float(o[5]),
                       __uint_as_float(o[6]), __uint_as_float(o[7]));
          if constexpr (decltype(is_q)::value) {
            rs += __shfl_xor_sync(0xffffffffu, rs, 1);
            rs += __shfl_xor_sync(0xffffffffu, rs, 2);
            if (su == 0) st_shared_u32(qsum_addr + row * 4, (uint32_t)rs);
          }
        }
      };
      int kr = 0, cq = 0;
      const Item im = decode(blockIdx.x);
      const int nt = im.nt, n = im.n;
      auto convert_q = [&](int t2) {
        mbar_wait(qraw_full, cq & 1);
        unpack_tile(sRawQ, sQ + t2 * QT, std::true_type{}, sQsum + t2 * 512);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) { mbar_arrive(q_full(t2)); mbar_arrive(qraw_empty); }
        ++cq;
      };
      if (n > 0) convert_q(0);
      for (int it = 0; it < n; ++it) {
        const int idx = 2 * it, s = idx % NS, rs = kr % NR;
        mbar_wait(raw_full(rs), (kr / NR) & 1);
        mbar_wait(kv_empty(s), ((idx / NS) & 1) ^ 1);
        unpack_tile(sRawK + rs * RAW, sKV + s * STG, std::false_type{}, 0u);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) { mbar_arrive(kv_full(s)); mbar_arrive(raw_empty(rs)); }
        ++kr;
        if (it == 0 && nt == 2) convert_q(1);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  // the allocating warp frees the columns, reading their address back from the slot: keeping `tmem` live through every role
  // costs a register that ptxas then finds by spilling (fp32 split kernel)
  if (warp == 9) tmem_dealloc(*reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw)), 512);
}

// ---- tile skipping under an external mask (north_star item 3): a two-kernel pre-pass reads the mask once and leaves, per
// (mask batch, mask head, query block of 256 rows), the compacted list of KV tiles that hold at least one visible element
// (bool: non-zero byte; additive: value > -inf) inside the block's causal / window range.
struct MaskTileParams {
  const void* mask;
  int kind, scalar;
  long long sb, sh, sq;
  int Sq, Skv, causal, window, nqb, nkt, MH;
  int* tiles;
  int* counts;
};

// per (KV tile, query block, mask batch x head): flag = the tile lies in the causal / window range of the block and holds at
// least one visible element (1), or is visible everywhere with a no-op mask (2).  Lane = column (4 coalesced loads per row).
// Two shapes of the same kernel, chosen by the tile count (launch_flags):
//   WARP_TILE = false: a CTA of 64 threads per tile, its two warps share the rows -- few tiles (a [1, 1, S, S] mask at the FLUX shape has
//     648): the latency chain of a tile that must be read in full (uniform tiles of a packing mask) is what counts, 29.5 us there
//     against 45.7 us with one warp per tile;
//   WARP_TILE = true: one warp per tile, 8 neighbouring KV tiles per CTA, no block-level synchronisation -- many tiles (dense
//     [1, H, S, S]: 15552, each decided by its first rows): the CTA launch rate bounds the pass, 25 us with a 256-thread CTA per tile,
//     20-24 us with 64-thread CTAs, 14-17 us with a warp per tile (profiles/r02bi_launches_mask.csv, r02bj_launches_mask.csv).
template <bool WARP_TILE>
__global__ void __launch_bounds__(WARP_TILE ? 256 : 64, WARP_TILE ? 4 : 16) mask_flags_kernel(const MaskTileParams q, uint8_t* __restrict__ flags) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j = WARP_TILE ? blockIdx.x * 8 + warp : blockIdx.x, qb = blockIdx.y, mbh = blockIdx.z;
  if (j >= q.nkt) return;                                  // (WARP_TILE only: whole warps, no barrier follows)
  const int mb = mbh / q.MH, mh = mbh % q.MH;
  const int r0 = qb * 256, rows = min(256, q.Sq - r0);
  constexpr int NW = WARP_TILE ? 1 : 2, RPW = 4;           // warps sharing a tile, rows per warp in the first round
  const int wt = WARP_TILE ? 0 : warp;                     // this warp's index among them
  int klo, khi;
  visible_key_range(q.causal, q.window, q.Skv, r0, min(r0 + 256, q.Sq), klo, khi);
  const int j_lo = klo >> 7, j_hi = khi > klo ? (khi + 127) >> 7 : j_lo;
  int any = 0, all = 1;         // any element visible / every element a no-op (bool: set; additive: exactly 0)
  if (j >= j_lo && j < j_hi) {
    const int c0 = j * 128, ncol = min(128, q.Skv - c0);
    const int nrows = q.sq ? rows : 1;                     // a mask broadcast over the rows: one row decides
    // a warp stops as soon as its rows prove the tile "partial" (something visible and something that is not a no-op): a dense
    // bias is decided by the first round of 4 rows per warp; tiles that look uniform are then read in rounds of 16 rows per warp
    // (64 loads in flight per lane)
    // two passes over raw[][]: first nothing but the loads (volatile asm: they stay back to back, all in flight together), then the
    // conversions -- fused into one loop the compiler pairs every load with its conversion and the round trips serialise (64 per
    // round: the two-phase version measured 70 us on a packing mask before this, profiles/r02bh_launches_mask.csv)
    const int esz_sel = q.kind == kMaskBool ? 0 : q.scalar == kMaskF32 ? 2 : 1;
    auto round = [&](int rb, auto nr_tag) {
      constexpr int NR = decltype(nr_tag)::value;
      uint32_t raw[NR][4];
#pragma unroll
      for (int i = 0; i < NR; ++i) {
        const int rr = min(rb + i, nrows - 1);             // past the end: the last row again
        const long long off = (long long)mb * q.sb + (long long)mh * q.sh + (long long)(r0 + rr) * q.sq + c0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const long long e = off + min(lane + 32 * k, ncol - 1);      // past the end: the last key again
          if (esz_sel == 0) raw[i][k] = ldg_pred_u8(reinterpret_cast<const uint8_t*>(q.mask) + e, true, 0u);
          else if (esz_sel == 2) raw[i][k] = ldg_pred_b32(reinterpret_cast<const float*>(q.mask) + e, true, 0u);
          else raw[i][k] = ldg_pred_u16(reinterpret_cast<const uint16_t*>(q.mask) + e, true, 0u);
        }
      }
#pragma unroll
      for (int i = 0; i < NR; ++i) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float val;
          if (esz_sel == 0) val = raw[i][k] != 0u ? 0.f : -CUDART_INF_F;
          else if (esz_sel == 2) val = __uint_as_float(raw[i][k]);
          else if (q.scalar == kMaskBF16) val = __uint_as_float(raw[i][k] << 16);
          else val = __half2float(__ushort_as_half((unsigned short)raw[i][k]));
          any |= val > -CUDART_INF_F;
          all &= val == 0.f;
        }
      }
      return __any_sync(0xffffffffu, any) && !__all_sync(0xffffffffu, all);
    };
    // full tiles whose rows are aligned for it take one vector load per row and lane (4 keys: 4 / 8 / 16 bytes) instead of four
    // element loads, and the row offset is one multiply-add on a hoisted base: the pre-pass of a dense [1, H, S, S] mask spent more
    // instructions on addresses than on loads
    const long long base_off = (long long)mb * q.sb + (long long)mh * q.sh + (long long)r0 * q.sq + c0;
    const int esz = esz_sel == 0 ? 1 : esz_sel == 2 ? 4 : 2;
    const uintptr_t base_addr = reinterpret_cast<uintptr_t>(q.mask) + (uintptr_t)(base_off * esz);
    const bool vec_ok = ncol == 128 && (base_addr & (uintptr_t)(4 * esz - 1)) == 0 && ((q.sq * esz) & (4 * esz - 1)) == 0;
    auto round_vec = [&](int rb, auto nr_tag, auto esz_tag) {
      constexpr int NR = decltype(nr_tag)::value, ESZ = decltype(esz_tag)::value, W = ESZ;      // words per lane and row: 1 / 2 / 4
      uint32_t raw[NR][W];
      const char* lane_ptr = reinterpret_cast<const char*>(base_addr) + lane * 4 * ESZ;
#pragma unroll
      for (int i = 0; i < NR; ++i) {
        const char* ptr = lane_ptr + (long long)min(rb + i, nrows - 1) * q.sq * ESZ;          // past the end: the last row again
        if constexpr (ESZ == 1) asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(raw[i][0]) : "l"(ptr));
        else if constexpr (ESZ == 2) asm volatile("ld.global.nc.v2.u32 {%0, %1}, [%2];" : "=r"(raw[i][0]), "=r"(raw[i][1]) : "l"(ptr));
        else asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(raw[i][0]), "=r"(raw[i][1]), "=r"(raw[i][2]), "=r"(raw[i][3]) : "l"(ptr));
      }
#pragma unroll
      for (int i = 0; i < NR; ++i) {
        if constexpr (ESZ == 1) {                          // four bool bytes: any byte set / no zero byte
          const uint32_t w = raw[i][0];
          any |= w != 0u;
          all &= ((w - 0x01010101u) & ~w & 0x80808080u) == 0u;
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float val;
            if constexpr (ESZ == 4) val = __uint_as_float(raw[i][k]);
            else {
              const uint32_t h16 = (raw[i][k >> 1] >> (16 * (k & 1))) & 0xffffu;
              val = q.scalar == kMaskBF16 ? __uint_as_float(h16 << 16) : __half2float(__ushort_as_half((unsigned short)h16));
            }
            any |= val > -CUDART_INF_F;
            all &= val == 0.f;
          }
        }
      }
      return __any_sync(0xffffffffu, any) && !__all_sync(0xffffffffu, all);
    };
    // rounds: first RPW rows per warp, then RPW2 rows per warp and round until the tile is decided or read
    auto walk = [&](auto first, auto later, int rpw2) {
      bool decided = false;
      if (wt * RPW < nrows) decided = first(wt * RPW);
      for (int rb = NW * RPW + wt * rpw2; rb < nrows && !decided; rb += NW * rpw2) decided = later(rb);
    };
    // (32 raw words per lane in the later rounds of every variant: the pass wants many resident warps)
    using I1 = std::integral_constant<int, 1>;
    using I2 = std::integral_constant<int, 2>;
    using I4 = std::integral_constant<int, 4>;
    using I8 = std::integral_constant<int, 8>;
    using I16 = std::integral_constant<int, 16>;
    using I32 = std::integral_constant<int, 32>;
    if (vec_ok && esz_sel == 0)
      walk([&](int rb) { return round_vec(rb, I4{}, I1{}); }, [&](int rb) { return round_vec(rb, I32{}, I1{}); }, 32);
    else if (vec_ok && esz_sel == 1)
      walk([&](int rb) { return round_vec(rb, I4{}, I2{}); }, [&](int rb) { return round_vec(rb, I16{}, I2{}); }, 16);
    else if (vec_ok)
      walk([&](int rb) { return round_vec(rb, I4{}, I4{}); }, [&](int rb) { return round_vec(rb, I8{}, I4{}); }, 8);
    else
      walk([&](int rb) { return round(rb, I4{}); }, [&](int rb) { return round(rb, I8{}); }, 8);
  }
  if constexpr (WARP_TILE) {
    any = __any_sync(0xffffffffu, any);
    all = __all_sync(0xffffffffu, all);
    if (lane == 0) flags[((size_t)mbh * q.nqb + qb) * q.nkt + j] = any ? (all ? 2 : 1) : 0;
  } else {
    any = __syncthreads_or(any);
    all = __syncthreads_and(all);
    if (threadIdx.x == 0) flags[((size_t)mbh * q.nqb + qb) * q.nkt + j] = any ? (all ? 2 : 1) : 0;
  }
}

// grid shape by tile count (see the kernel)
template <typename M>
void launch_flags(const MaskTileParams& q, const M& m, uint8_t* flags, cudaStream_t st) {
  const long long tiles = (long long)m.nkt * m.nqb * m.MB * m.MH;
  if (tiles >= 4096)
    mask_flags_kernel<true><<<dim3((unsigned)((m.nkt + 7) / 8), (unsigned)m.nqb, (unsigned)(m.MB * m.MH)), 256, 0, st>>>(q, flags);
  else
    mask_flags_kernel<false><<<dim3((unsigned)m.nkt, (unsigned)m.nqb, (unsigned)(m.MB * m.MH)), 64, 0, st>>>(q, flags);
}

// one thread per list: compacts the flagged tile indices in ascending order; kTileNoMask marks tiles on which the mask is a
// no-op (all attend / all zero), so the attention kernel neither loads nor applies it there
__global__ void mask_compact_kernel(const uint8_t* __restrict__ flags, int* __restrict__ tiles, int* __restrict__ counts,
                                    int lists, int nkt) {
  const int lid = blockIdx.x * blockDim.x + threadIdx.x;
  if (lid >= lists) return;
  int cnt = 0;
  for (int j = 0; j < nkt; ++j)
    if (const int f = flags[(size_t)lid * nkt + j]) tiles[(size_t)lid * nkt + cnt++] = j | (f == 2 ? kTileNoMask : 0);
  counts[lid] = cnt;
}

// ------------------------------------------------------------------------------------------------ host side
using tc::encode_fn;
using tc::make_map;

bool view_ok(const TensorView& t, int64_t, int64_t Hn, int64_t B) { return tc::view_ok(t, Hn, B); }

template <int D, int MODE, int MASKED>
cudaError_t launch_k(const FwdTcParams& prm, dim3 grid, cudaStream_t st) {
  static bool attr_set = false;
  auto kern = fwd_tc_kernel<D, MODE, MASKED>;
  constexpr int kSmem = Cfg<D, MODE, MASKED>::kSmem;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  kern<<<grid, kThreads, kSmem, st>>>(prm);
  return cudaGetLastError();
}

// dense 1- / 2-byte masks take the instantiation that stages mask tiles in shared memory (where the mode has one)
template <int D, int MODE>
cudaError_t launch(const FwdTcParams& prm, dim3 grid, cudaStream_t st) {
  if (!prm.mask) return launch_k<D, MODE, 0>(prm, grid, st);
  if constexpr (Cfg<D, MODE, 2>::kMaskTma) {
    if (prm.mask_tma) return launch_k<D, MODE, 2>(prm, grid, st);
  }
  return launch_k<D, MODE, 1>(prm, grid, st);
}

}  // namespace

cudaError_t launch_fwd_tc_kernel(const FwdTcParams& prm_in, int D, int mode, cudaStream_t st, int B) {
  FwdTcParams prm = prm_in;
  prm.nbatch = B;
  ptx::watchdog_bind();
  const bool wide = mode == kFwdWideF16 || mode == kFwdWideBF16;
  const long long items = prm.kv_len ? (prm.kv_slots ? (long long)prm.kv_slots : (long long)prm.kv_nqi * B) * prm.kv_nsplit * prm.Hkv
                                     : (long long)((prm.Sq + 255) / 256) * prm.H * B * (wide ? 2 : 1);
  if (items <= 0 || items > 0x7fffffffLL) return cudaErrorInvalidValue;
  const dim3 grid((unsigned)items, 1, 1);        // one CTA per work item
  if (wide) {                                    // D is the head dim of the problem (256); the kernel's tiles are 128 wide
    if (D != 256) return cudaErrorInvalidValue;
    return mode == kFwdWideBF16 ? launch<128, kFwdWideBF16>(prm, grid, st) : launch<128, kFwdWideF16>(prm, grid, st);
  }
  if (D == 64 && mode == kFwdBF16) return launch<64, kFwdBF16>(prm, grid, st);
  if (D == 64 && mode == kFwdF16) return launch<64, kFwdF16>(prm, grid, st);
  if (D != 128) return cudaErrorInvalidValue;
  switch (mode) {
    case kFwdF16: return launch<128, kFwdF16>(prm, grid, st);
    case kFwdBF16: return launch<128, kFwdBF16>(prm, grid, st);
    case kFwdI8: return launch<128, kFwdI8>(prm, grid, st);
    case kFwdI8F8: return launch<128, kFwdI8F8>(prm, grid, st);
    case kFwdSplit: return launch<128, kFwdSplit>(prm, grid, st);
    case kFwdI4: return launch<128, kFwdI4>(prm, grid, st);
    case kFwdI4F8: return launch<128, kFwdI4F8>(prm, grid, st);
    default: return cudaErrorInvalidValue;
  }
}

// external masks the tensor-core forward reads itself: keys contiguous (the row of a tile is one 128-element run)
bool fwd_tc_mask_ok(const AttnParams& p) {
  return p.mask_kind == kMaskNone || !p.mask || p.mask_sk == 1;
}

void fwd_tc_set_mask(FwdTcParams& prm, const AttnParams& p) {
  prm.mask_tma = 0;
  if (p.mask_kind == kMaskNone || !p.mask) return;
  prm.mask = p.mask; prm.mask_kind = p.mask_kind; prm.mask_scalar = p.mask_scalar;
  prm.mask_sb = p.mask_sb; prm.mask_sh = p.mask_sh; prm.mask_sq = p.mask_sq;
  // dense masks (one row of terms per query row) with 1- or 2-byte elements are staged through shared memory by TMA
  // (tc::make_mask_map); masks broadcast over the rows (key padding) and fp32 terms (64 KB per tile) keep the in-place reads
  if (tc::make_mask_map(&prm.tm, p))
    prm.mask_tma = 1;
}

namespace {
struct MaskLists { long long lists; int nqb, nkt, MB, MH; };
MaskLists mask_lists(const AttnParams& p) {
  MaskLists m;
  m.nqb = (p.Sq + 255) / 256; m.nkt = (p.Skv + 127) / 128;
  m.MB = p.mask_sb ? p.B : 1; m.MH = p.mask_sh ? p.H : 1;
  m.lists = (long long)m.MB * m.MH * m.nqb;
  return m;
}
}  // namespace

size_t fwd_tc_mask_scratch_bytes(const AttnParams& p) {
  if (p.mask_kind == kMaskNone || !p.mask || getenv("MFA_DISABLE_MASK_SKIP")) return 0;
  const MaskLists m = mask_lists(p);
  return (size_t)m.lists * (m.nkt + 1) * sizeof(int) + (size_t)m.lists * m.nkt + 16;      // counts, lists, flags
}

// Tile classification shared with the backward (attn_bwd_tc.cu): flags[((mb * MH + mh) * nqb + qb) * nkt + j] = 0 hidden,
// 1 partial, 2 no-op for query block qb (256 rows) x KV tile j (128 keys).
void mask_tile_dims(const AttnParams& p, int& nqb, int& nkt, int& MB, int& MH) {
  const MaskLists m = mask_lists(p);
  nqb = m.nqb; nkt = m.nkt; MB = m.MB; MH = m.MH;
}

cudaError_t launch_mask_flags(const AttnParams& p, uint8_t* flags, cudaStream_t st) {
  const MaskLists m = mask_lists(p);
  if (m.lists > 0x3fffffffLL || m.MB * (long long)m.MH > 65535 || m.nqb > 65535) return cudaErrorInvalidValue;
  MaskTileParams q;
  q.mask = p.mask; q.kind = p.mask_kind; q.scalar = p.mask_scalar;
  q.sb = p.mask_sb; q.sh = p.mask_sh; q.sq = p.mask_sq;
  q.Sq = p.Sq; q.Skv = p.Skv; q.causal = p.causal; q.window = p.window; q.nqb = m.nqb; q.nkt = m.nkt; q.MH = m.MH;
  q.counts = nullptr; q.tiles = nullptr;
  launch_flags(q, m, flags, st);
  ++g_launch_count;
  return cudaGetLastError();
}

// Builds the visible-tile lists into p.mask_tile_scratch (when given) and points the kernel parameters at them.
cudaError_t fwd_tc_build_mask_tiles(FwdTcParams& prm, const AttnParams& p, cudaStream_t st) {
  prm.mtiles = nullptr; prm.mcounts = nullptr; prm.m_nkt = 0;
  if (!prm.mask || !p.mask_tile_scratch || fwd_tc_mask_scratch_bytes(p) == 0) return cudaSuccess;
  const MaskLists m = mask_lists(p);
  if (m.lists > 0x3fffffffLL || m.MB * (long long)m.MH > 65535 || m.nqb > 65535) return cudaSuccess;   // visit every tile
  MaskTileParams q;
  q.mask = p.mask; q.kind = p.mask_kind; q.scalar = p.mask_scalar;
  q.sb = p.mask_sb; q.sh = p.mask_sh; q.sq = p.mask_sq;
  q.Sq = p.Sq; q.Skv = p.Skv; q.causal = p.causal; q.window = p.window; q.nqb = m.nqb; q.nkt = m.nkt; q.MH = m.MH;
  q.counts = p.mask_tile_scratch;
  q.tiles = p.mask_tile_scratch + m.lists;
  uint8_t* flags = reinterpret_cast<uint8_t*>(q.tiles + m.lists * m.nkt);
  launch_flags(q, m, flags, st);
  mask_compact_kernel<<<(unsigned)((m.lists + 127) / 128), 128, 0, st>>>(flags, q.tiles, q.counts, (int)m.lists, m.nkt);
  g_launch_count += 2;
  prm.mtiles = q.tiles; prm.mcounts = q.counts; prm.m_nkt = m.nkt;
  return cudaGetLastError();
}

// O (fp32, or bf16 / fp16 on request) goes out through TMA bulk stores from a swizzled staging tile (coalesced, asynchronous)
// when the view allows a tensor map; otherwise (and in the accumulate mode) the row-owner threads store directly.
void fwd_tc_set_out_map(FwdTcParams& prm, const AttnParams& p) {
  prm.o_tma = 0;
  if (p.accumulate || getenv("MFA_DISABLE_TMA_STORE")) return;
  if (p.o_dtype != kF32 && p.o_dtype != kBF16 && p.o_dtype != kF16) return;
  if (!tc::view_ok(p.o, p.H, p.B, dtype_bytes(p.o_dtype))) return;
  if (tc::make_map(&prm.to, p.o, p.o_dtype, p.B, p.H, p.Sq, p.D)) prm.o_tma = 1;
}

bool fwd_tc_eligible(const AttnParams& p) {
  if (getenv("MFA_DISABLE_TC")) return false;
  if (p.in_dtype != kBF16 && p.in_dtype != kF16) return false;
  // head dims 64 / 128 / 256 run as they are; any other multiple of 8 up to 256 runs on the next kernel width with the missing
  // columns zero-filled by TMA on the way in (tensor extent < box extent) and left out on the way out (the TMA store clips
  // them, the direct stores stop at FwdTcParams::dv)
  if (p.D < 8 || p.D > 256 || (p.D & 7)) return false;
  if (p.D > 128 && p.accumulate) return false;
  if (!fwd_tc_mask_ok(p)) return false;
  if (!(p.scale > 0.f) || p.Sq <= 0 || p.Skv <= 0 || p.B <= 0 || p.H <= 0 || p.Hkv <= 0 || p.H % p.Hkv) return false;
  if (p.B > 65535 || p.H > 65535) return false;
  if (!view_ok(p.q, p.Sq, p.H, p.B) || !view_ok(p.k, p.Skv, p.Hkv, p.B) || !view_ok(p.v, p.Skv, p.Hkv, p.B)) return false;
  if (p.o.sd != 1) return false;
  const int oes = dtype_bytes(p.o_dtype);
  if ((reinterpret_cast<uintptr_t>(p.o.ptr) & 15) || ((p.o.ss * oes) & 15) || ((p.o.sh * oes) & 15) || ((p.o.sb * oes) & 15))
    return false;
  return encode_fn() != nullptr;
}

cudaError_t launch_fwd_tc(const AttnParams& p, cudaStream_t st) {
  FwdTcParams prm = {};
  if (!make_map(&prm.tq, p.q, p.in_dtype, p.B, p.H, p.Sq, p.D) || !make_map(&prm.tk, p.k, p.in_dtype, p.B, p.Hkv, p.Skv, p.D) ||
      !make_map(&prm.tv, p.v, p.in_dtype, p.B, p.Hkv, p.Skv, p.D))
    return cudaErrorInvalidValue;
  prm.o = const_cast<void*>(p.o.ptr);
  prm.o_sb = p.o.sb; prm.o_sh = p.o.sh; prm.o_ss = p.o.ss;
  prm.lse = p.lse;
  prm.lse_sh = p.lse_sh > 0 ? p.lse_sh : p.Sq;
  prm.accumulate = p.accumulate && p.lse && p.o_dtype == kF32;
  prm.o_dtype = p.o_dtype;
  prm.H = p.H; prm.Hkv = p.Hkv; prm.Sq = p.Sq; prm.Skv = p.Skv;
  prm.c = p.scale * kLog2e;
  prm.causal = p.causal; prm.window = p.window;
  prm.cu_q = p.cu_q; prm.cu_k = p.cu_k; prm.nseq = p.nseq;
  fwd_tc_set_out_map(prm, p);
  fwd_tc_set_mask(prm, p);
  if (cudaError_t me = fwd_tc_build_mask_tiles(prm, p, st); me != cudaSuccess) return me;
  const bool bf = p.in_dtype == kBF16;
  const int Dk = p.D <= 64 ? 64 : p.D <= 128 ? 128 : 256;          // kernel width (zero-padded head dims: see fwd_tc_eligible)
  prm.dv = p.D;
  if (Dk == 256) {
    cudaError_t e = launch_fwd_tc_kernel(prm, Dk, bf ? kFwdWideBF16 : kFwdWideF16, st, p.B);
    g_last_kernel = prm.mask ? (bf ? "fwd_tc_bf16_d256_mask" : "fwd_tc_fp16_d256_mask") : (bf ? "fwd_tc_bf16_d256" : "fwd_tc_fp16_d256");
    ++g_launch_count;
    return e;
  }
  cudaError_t e = launch_fwd_tc_kernel(prm, Dk, bf ? kFwdBF16 : kFwdF16, st, p.B);
  if (prm.mask && prm.mask_tma)       // dense 1- / 2-byte mask staged in shared memory by TMA
    g_last_kernel = Dk == 128 ? (bf ? "fwd_tc_bf16_d128_tma_mask" : "fwd_tc_fp16_d128_tma_mask") : (bf ? "fwd_tc_bf16_d64_tma_mask" : "fwd_tc_fp16_d64_tma_mask");
  else if (Dk == 128) g_last_kernel = prm.mask ? (bf ? "fwd_tc_bf16_d128_mask" : "fwd_tc_fp16_d128_mask") : (bf ? "fwd_tc_bf16_d128" : "fwd_tc_fp16_d128");
  else g_last_kernel = prm.mask ? (bf ? "fwd_tc_bf16_d64_mask" : "fwd_tc_fp16_d64_mask") : (bf ? "fwd_tc_bf16_d64" : "fwd_tc_fp16_d64");
  ++g_launch_count;
  return e;
}

// ------------------------------------------------------------------------------------------------ decode over a K/V cache
namespace {

struct KvcCombine {
  const float* o_part;       // [items][2][rows][D]
  const float* l_part;       // [items][2][rows]
  void* o;
  long long o_sb, o_sh, o_ss;
  int o_dtype;
  float* lse;                // [B, H, Sq], or [H, total_q] with cu_q
  const int* cu_q;           // KvCacheParams::cu_q
  int H, Hkv, Sq, D, G, sqb, rows, nqi, nsplit, slots;
  int nseq, nrows;           // sequences, and query rows per grid z (Sq, or total_q with cu_q)
};

// One warp per query row t of sequence z (without cu_q) or of the packed rows (with cu_q, whose sequence a binary search finds),
// grid (nrows / 8, H, B or 1): merges the row's partials of every split (lse_merge_*), writes O in the output's type and stride
// and L.  Splits without a visible key (L_k = -inf) are not read; rows of no sequence are not written, and rows of a sequence
// past Sq (max_seqlen_q) get O = +0, L = -inf.  Lane i holds head dims [4i, 4i + 4).
__global__ void __launch_bounds__(256) kvcache_combine_kernel(const KvcCombine c) {
  const int t = blockIdx.x * 8 + (threadIdx.x >> 5), h = blockIdx.y, z = blockIdx.z;
  const int lane = threadIdx.x & 31;
  if (t >= c.nrows) return;
  int b = z, s = t;
  if (c.cu_q) {
    b = segment_of(c.cu_q, c.nseq, t);
    const int q0 = seg_offset(c.cu_q, b, c.nrows);
    if (t < q0 || t >= seg_offset(c.cu_q, b + 1, c.nrows)) return;
    s = t - q0;
  }
  const long long rid = ((long long)z * c.H + h) * c.nrows + t;
  const int hk = h / c.G, chunk = s / c.sqb;
  const int r = (h % c.G) * c.sqb + s % c.sqb;
  // the items of this row's query item, split k at item0 + k * step (KvCachePlan: per-sequence or packed slots)
  const long long item0 = c.slots ? (long long)hk * c.nsplit * c.slots + kvc_first_slot(c.cu_q, b, c.nrows, 2 * c.sqb) + (chunk >> 1)
                                  : ((long long)b * c.Hkv + hk) * c.nsplit * c.nqi + (chunk >> 1);
  const int step = c.slots ? c.slots : c.nqi;
  auto slot = [&](int k) { return ((item0 + (long long)k * step) * 2 + (chunk & 1)) * c.rows + r; };
  const int nk = s < c.Sq ? c.nsplit : 0;
  float m = -CUDART_INF_F;
  for (int k = lane; k < nk; k += 32) m = fmaxf(m, __ldg(c.l_part + slot(k)));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float4 acc = make_float4(-0.f, -0.f, -0.f, -0.f);       // -0 + x == x for every x: one split passes through unchanged
  float L = -CUDART_INF_F;
  const int c0 = lane * 4;
  if (m != -CUDART_INF_F) {
    float wsum = 0.f;
    for (int k = lane; k < nk; k += 32) wsum += lse_merge_weight(__ldg(c.l_part + slot(k)), m);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
    L = lse_merge_total(m, wsum);
    for (int k = 0; k < nk; ++k) {
      const float lk = __ldg(c.l_part + slot(k));
      if (lk == -CUDART_INF_F || c0 >= c.D) continue;
      const float wk = lse_merge_weight(lk, m) / wsum;
      const float4 ok = __ldg(reinterpret_cast<const float4*>(c.o_part + slot(k) * c.D + c0));
      acc = make_float4(fmaf(wk, ok.x, acc.x), fmaf(wk, ok.y, acc.y), fmaf(wk, ok.z, acc.z), fmaf(wk, ok.w, acc.w));
    }
  }
  if (m == -CUDART_INF_F) acc = make_float4(0.f, 0.f, 0.f, 0.f);   // a row without keys: O = +0
  if (c0 < c.D) {
    const long long off = (long long)z * c.o_sb + (long long)h * c.o_sh + (long long)t * c.o_ss + c0;
    auto put = [&](int i, float x) {
      if (c.o_dtype == kF32) reinterpret_cast<float*>(c.o)[off + i] = x;
      else reinterpret_cast<uint16_t*>(c.o)[off + i] = (uint16_t)((c.o_dtype == kBF16 ? pack_bf16(x, 0.f) : pack_f16(x, 0.f)) & 0xffffu);
    };
    put(0, acc.x); put(1, acc.y); put(2, acc.z); put(3, acc.w);
  }
  if (lane == 0 && c.lse) c.lse[rid] = L;
}

}  // namespace

KvCachePlan kvcache_plan(const KvCacheParams& p, int sm_count) {
  KvCachePlan k;
  k.G = p.H / p.Hkv;
  k.sqb = std::min(p.Sq, 128 / k.G);
  k.rows = k.G * k.sqb;
  const int chunks = (p.Sq + k.sqb - 1) / k.sqb;
  k.nqi = (chunks + 1) / 2;
  // query-item slots per KV head and split: nqi per sequence, or with per-sequence token counts the packed slots when fewer
  long long slots = (long long)p.B * k.nqi;
  k.slots = 0;
  if (p.cu_q) {
    const long long packed = p.total_q / (2 * k.sqb) + p.B;
    if (packed < slots) slots = k.slots = (int)packed;
  }
  // split the keys when the items of the call leave SMs idle: about one wave of CTAs, each split at least two 128-key tiles
  const long long base = slots * p.Hkv;
  const int ntiles = (p.cap + 127) / 128;
  long long ns = base < sm_count ? sm_count / base : 1;
  ns = std::max(1LL, std::min(ns, (long long)ntiles / 2));
  const int per = (int)((ntiles + ns - 1) / ns);
  k.nsplit = (ntiles + per - 1) / per;                   // no split is left without tiles
  k.items = base * k.nsplit;
  k.o_bytes = ((size_t)k.items * 2 * k.rows * p.D * sizeof(float) + 255) & ~(size_t)255;
  k.l_bytes = (size_t)k.items * 2 * k.rows * sizeof(float);
  return k;
}

cudaError_t launch_fwd_kvcache(const KvCacheParams& p, const KvCachePlan& k, void* scratch, cudaStream_t st) {
  if (k.items <= 0 || k.items > 0x7fffffffLL || p.H > 65535 || p.B > 65535) return cudaErrorInvalidValue;   // (combine grid y / z)
  float* o_part = reinterpret_cast<float*>(scratch);
  float* l_part = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(scratch) + k.o_bytes);
  FwdTcParams prm = {};
  const int Dk = p.D <= 64 ? 64 : 128;
  const bool paged = p.block_table != nullptr;
  TensorView kv[2] = {p.k, p.v};
  int kB = p.B, kS = p.cap, box = 128;
  if (paged) {                                 // [num_pages, page_size, Hkv, D] pools seen as [B = pages, H = Hkv, S = page, D]
    for (TensorView& t : kv) { t.sb = (int64_t)p.page_size * p.Hkv * p.D; t.sh = p.D; t.ss = (int64_t)p.Hkv * p.D; t.sd = 1; }
    kB = p.num_pages; kS = p.page_size;
    box = std::gcd(p.page_size, 128);
  }
  const TensorView ov = {o_part, 2LL * k.rows * p.D, (int64_t)k.rows * p.D, p.D, 1};
  const bool packed_q = p.cu_q != nullptr;      // Q as [1, H, total_q, D]
  if (!tc::make_map_gqa(&prm.tq, p.q, p.in_dtype, packed_q ? 1 : p.B, p.Hkv, k.G, packed_q ? p.total_q : p.Sq, p.D, k.sqb) ||
      !make_map(&prm.tk, kv[0], p.in_dtype, kB, p.Hkv, kS, p.D, box) || !make_map(&prm.tv, kv[1], p.in_dtype, kB, p.Hkv, kS, p.D, box) ||
      !make_map(&prm.to, ov, kF32, (int)k.items, 2, k.rows, p.D, k.rows))
    return cudaErrorInvalidValue;
  prm.o_tma = 1;
  prm.o_dtype = kF32;
  prm.lse = l_part;
  prm.H = p.H; prm.Hkv = p.Hkv; prm.Sq = p.Sq; prm.Skv = p.cap;
  prm.dv = p.D;
  prm.c = p.scale * kLog2e;
  prm.causal = p.causal; prm.window = p.window;
  prm.kv_len = p.seqlens; prm.kv_pages = p.block_table;
  prm.kv_cap = p.cap; prm.kv_page = p.page_size; prm.kv_npages = p.num_pages;
  prm.kv_npb = paged ? p.cap / p.page_size : 0; prm.kv_box = box;
  prm.kv_g = k.G; prm.kv_sqb = k.sqb; prm.kv_rows = k.rows; prm.kv_nqi = k.nqi; prm.kv_nsplit = k.nsplit;
  prm.kv_qbytes = (Dk / 64) * 128 * k.rows;
  prm.kv_cu_q = p.cu_q; prm.kv_total = p.total_q; prm.kv_slots = k.slots;
  const bool bf = p.in_dtype == kBF16;
  cudaError_t e = launch_fwd_tc_kernel(prm, Dk, bf ? kFwdBF16 : kFwdF16, st, p.B);
  if (e != cudaSuccess) return e;
  KvcCombine c;
  c.o_part = o_part; c.l_part = l_part;
  c.o = const_cast<void*>(p.o.ptr); c.o_sb = p.o.sb; c.o_sh = p.o.sh; c.o_ss = p.o.ss; c.o_dtype = p.o_dtype;
  c.lse = p.lse;
  c.cu_q = p.cu_q;
  c.H = p.H; c.Hkv = p.Hkv; c.Sq = p.Sq; c.D = p.D; c.G = k.G; c.sqb = k.sqb; c.rows = k.rows; c.nqi = k.nqi; c.nsplit = k.nsplit;
  c.slots = k.slots; c.nseq = p.B; c.nrows = packed_q ? p.total_q : p.Sq;
  kvcache_combine_kernel<<<dim3((unsigned)((c.nrows + 7) / 8), (unsigned)p.H, packed_q ? 1u : (unsigned)p.B), 256, 0, st>>>(c);
  static const char* names[2][2][2] = {{{"fwd_tc_fp16_d64_kvcache", "fwd_tc_fp16_d64_kvcache_split"},
                                        {"fwd_tc_fp16_d128_kvcache", "fwd_tc_fp16_d128_kvcache_split"}},
                                       {{"fwd_tc_bf16_d64_kvcache", "fwd_tc_bf16_d64_kvcache_split"},
                                        {"fwd_tc_bf16_d128_kvcache", "fwd_tc_bf16_d128_kvcache_split"}}};
  g_last_kernel = names[bf][Dk == 128][k.nsplit > 1];
  g_launch_count += 2;
  return cudaGetLastError();
}

}  // namespace mfa
