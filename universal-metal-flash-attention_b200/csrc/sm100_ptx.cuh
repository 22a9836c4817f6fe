// sm100_ptx.cuh -- thin inline-PTX wrappers for the Blackwell (sm_100a) primitives the attention kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (TMEM alloc / ld / st / mma / commit), descriptors.
// Encodings follow the PTX ISA and were cross-checked against cute/arch/mma_sm100_desc.hpp (bit layouts only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mfa {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Spin until the phase with the given parity has completed.  Builds with -DMFA_MBAR_WATCHDOG (MFA_WATCHDOG=1 at build time)
// add a wall-clock watchdog that turns a protocol bug into a diagnosable trap instead of a hung GPU: after kWatchdogNs of
// %globaltimer in ONE wait the thread writes (block, thread, barrier address, parity) into a host-mapped record buffer
// (g_watchdog_log, set by the launcher; survives the dead context) and, after twice that time, traps.  The limit is seconds,
// so compute-sanitizer, a debugger or MPS time-slicing do not trip it.  Release builds spin without a limit.
#ifdef MFA_MBAR_WATCHDOG
constexpr unsigned long long kWatchdogNs = 3000000000ull;
struct WatchdogLog { unsigned int count; unsigned int pad; unsigned int rec[1024][4]; };
static __device__ WatchdogLog* g_watchdog_log = nullptr;      // one per translation unit and device: watchdog_bind()
// out of line on purpose: the hot wait loops (MMA issuer, softmax) must stay small in the instruction cache
static __device__ __noinline__ void watchdog_tick(uint32_t bar, uint32_t parity, unsigned long long& t0, bool& logged) {
  unsigned long long now;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
  if (t0 == 0) { t0 = now; return; }
  if (!logged && now - t0 > kWatchdogNs) {
    logged = true;
    if (WatchdogLog* lg = g_watchdog_log) {
      const unsigned int i = atomicAdd(&lg->count, 1u);
      if (i < 1024) {
        lg->rec[i][0] = blockIdx.x; lg->rec[i][1] = threadIdx.x; lg->rec[i][2] = bar; lg->rec[i][3] = parity;
        __threadfence_system();
      }
    }
  }
  if (now - t0 > 2 * kWatchdogNs) { asm volatile("trap;"); }
}
}  // namespace ptx
void* watchdog_device_log();          // ffi.cu: host-mapped record buffer (device view), allocated on first use
namespace ptx {
// called by a launcher before its first launch on the current device: points this translation unit's log pointer at the buffer
inline void watchdog_bind() {
  static bool done[64] = {false};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || done[dev]) return;
  void* d = watchdog_device_log();
  if (d && cudaMemcpyToSymbol(g_watchdog_log, &d, sizeof(d)) == cudaSuccess) done[dev] = true;
  else cudaGetLastError();
}
#else
inline void watchdog_bind() {}
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
#ifdef MFA_MBAR_WATCHDOG
  uint32_t spins = 0;
  unsigned long long t0 = 0;
  bool logged = false;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 4095u) == 0) watchdog_tick(bar, parity, t0, logged);
  }
#else
  while (!mbar_try_wait(bar, parity)) {}
#endif
}

// Long waits off the critical path (the epilogue warpgroup waiting a whole work item for its statistics): sleep between polls so
// the waiting warp does not compete for issue slots with the warps doing the work.
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
#ifdef MFA_MBAR_WATCHDOG
  unsigned long long t0 = 0;
  uint32_t spins = 0;
  bool logged = false;
#endif
  while (!mbar_try_wait(bar, parity)) {
    asm volatile("nanosleep.u32 256;" ::: "memory");
#ifdef MFA_MBAR_WATCHDOG
    if ((++spins & 1023u) == 0) watchdog_tick(bar, parity, t0, logged);
#endif
  }
}

// ------------------------------------------------------------------------------------------------ TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 4-D tiled load: coordinates innermost first (c0 = element in row, c1 = row, c2 = head, c3 = batch)
__device__ __forceinline__ void tma_load_4d(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// the same load with an L2 eviction policy (streams that are read once: evict-first)
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_normal() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_load_4d_hint(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                                 int c3, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(policy)
      : "memory");
}

// 5-D tiled load (ring attention: c4 = visiting slot)
__device__ __forceinline__ void tma_load_5d(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// flag polling for data written by another stream / GPU, followed by TMA reads of that data
__device__ __forceinline__ uint32_t ld_acquire_gpu_u32(const unsigned int* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void nanosleep_ns(uint32_t ns) { asm volatile("nanosleep.u32 %0;" ::"r"(ns) : "memory"); }
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// 4-D tiled store shared -> global (bulk async group); rows / columns outside the tensor are clipped by the TMA unit
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, uint32_t src_smem, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src_smem), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed bulk groups of this thread have finished READING their shared-memory source
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... all but the most recent one (a two-buffer staging ring: the buffer about to be refilled is free)
__device__ __forceinline__ void bulk_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
// all committed bulk groups of this thread are complete (writes performed)
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (TMA)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void st_shared_v4(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void ld_shared_v4(uint32_t addr, float& a, float& b, float& c, float& d) {
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a), "=f"(b), "=f"(c), "=f"(d) : "r"(addr) : "memory");
}
__device__ __forceinline__ void st_shared_v2(uint32_t addr, float a, float b) {
  asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void ld_shared_v2(uint32_t addr, float& a, float& b) {
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(a), "=f"(b) : "r"(addr) : "memory");
}
__device__ __forceinline__ void st_shared_u32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_shared_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_shared_u16(uint32_t addr) {
  uint16_t v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_shared_u8(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}

// 256-bit read-only global load (LDG.E.256 on sm_100): one full 32-byte sector per thread per request.  L1::no_allocate: the
// attention kernels carve ~225 KB of the 228 KB L1 / shared array out as shared memory, and the few KB of L1 left cap the
// lines in flight -- streaming mask rows past it took the dense fp32 mask forward from 0.76 to 0.56 ms at the FLUX shape
__device__ __forceinline__ void ldg256(const void* p, uint32_t* r) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "l"(p));
}

// predicated read-only scalar loads as volatile asm: a run of them stays a run of loads (the compiler otherwise re-fuses
// "load all, then convert all" into load-4 / convert-4 groups and the requests never overlap)
__device__ __forceinline__ uint32_t ldg_pred_b32(const void* p, bool pred, uint32_t dflt) {
  uint32_t v = dflt;
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.global.nc.b32 %0, [%1];\n\t}" : "+r"(v) : "l"(p), "r"((int)pred));
  return v;
}
__device__ __forceinline__ uint32_t ldg_pred_u16(const void* p, bool pred, uint32_t dflt) {
  unsigned short v = (unsigned short)dflt;
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.global.nc.u16 %0, [%1];\n\t}" : "+h"(v) : "l"(p), "r"((int)pred));
  return v;
}
__device__ __forceinline__ uint32_t ldg_pred_u8(const void* p, bool pred, uint32_t dflt) {
  uint32_t v = dflt;
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.global.nc.u8 %0, [%1];\n\t}" : "+r"(v) : "l"(p), "r"((int)pred));
  return v;
}

// 256-bit coherent global load / store (read-modify-write epilogues)
__device__ __forceinline__ void ld_global_v8(const float* p, float* r) {
  asm volatile("ld.global.L1::no_allocate.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]), "=f"(r[4]), "=f"(r[5]), "=f"(r[6]), "=f"(r[7])
               : "l"(p) : "memory");
}
__device__ __forceinline__ void st_global_v8(float* p, const float* r) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"l"(p), "f"(r[0]), "f"(r[1]), "f"(r[2]), "f"(r[3]), "f"(r[4]), "f"(r[5]), "f"(r[6]), "f"(r[7]) : "memory");
}

// 128-bit coherent global load / store (the forward's coalesced write-out / merge of O)
__device__ __forceinline__ float4 ld_global_v4(const void* p) {
  float4 r;
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ void st_global_v4(void* p, float a, float b, float c, float d) {
  asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// Named barriers (ids 1..15; id 0 is __syncthreads)
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ------------------------------------------------------------------------------------------------ tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]      (both operands through shared-memory descriptors)
__device__ __forceinline__ void mma_f16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accum)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]      (A read from tensor memory: P never leaves TMEM)
__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accum)
      : "memory");
}
// int8 x int8 -> int32
__device__ __forceinline__ void mma_i8_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accum)
      : "memory");
}
// fp8 (e4m3/e5m2) operands
__device__ __forceinline__ void mma_f8_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void mma_f8_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accum)
      : "memory");
}
// ---- warp-uniform issue path.  The whole MMA warp runs the issue loop in uniform control flow and one elected lane
// executes the instruction; descriptors arrive as (lo, hi) 32-bit halves so the per-MMA address update is a single
// uniform add.  (Issuing from inside `if (lane == 0)` makes ptxas wrap every UTCHMMA in an ELECT/BRA.U.ANY waterfall
// plus R2UR moves, ~15 dependent instructions per MMA -- slower than the 64-clock MMA itself; tools/mma_probe.cu.)
__device__ __forceinline__ void mma_f16_ss_u(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                             uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p, pe;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void mma_f16_ts_u(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                             uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p, pe;\n\t.reg .b64 db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void mma_i8_ss_u(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                            uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p, pe;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe tcgen05.mma.cta_group::1.kind::i8 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void mma_f8_ts_u(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                            uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p, pe;\n\t.reg .b64 db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], [%1], db, %4, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void tc_commit_u(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar)
      : "memory");
}
// SWIZZLE_128B descriptor halves: hi = SBO (1024 B between 8-row groups) | version 1 | layout 2; lo = addr>>4 | LBO>>4<<16.
constexpr uint32_t kDescHiSw128 = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) { return (saddr >> 4) | ((lbo_bytes >> 4) << 16); }

// Arrive on an mbarrier once every tcgen05 operation issued so far by this thread has completed.
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// Shared-memory matrix descriptor (64-bit): [0,14) addr>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version = 1,
// [61,64) layout (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | (2ull << 61);
}

// Instruction descriptor (32-bit), kind::f16 / kind::i8 / kind::f8f6f4:
// [4,6) D format (1 = f32, 2 = s32), [7,10) A format, [10,13) B format, [15] A major, [16] B major (1 = MN-major),
// [17,23) N>>3, [24,29) M>>4.
__host__ __device__ constexpr uint32_t make_idesc(uint32_t dfmt, uint32_t afmt, uint32_t bfmt, uint32_t a_mn, uint32_t b_mn,
                                                  uint32_t M, uint32_t N) {
  return (dfmt << 4) | (afmt << 7) | (bfmt << 10) | (a_mn << 15) | (b_mn << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// TMEM <-> registers, shape 32x32b: lane i of the warp owns TMEM lane (base_lane + i); xN = N consecutive columns.
#define MFA_R8(r, o) "=r"(r[o + 0]), "=r"(r[o + 1]), "=r"(r[o + 2]), "=r"(r[o + 3]), "=r"(r[o + 4]), "=r"(r[o + 5]), "=r"(r[o + 6]), "=r"(r[o + 7])
#define MFA_W8(r, o) "r"(r[o + 0]), "r"(r[o + 1]), "r"(r[o + 2]), "r"(r[o + 3]), "r"(r[o + 4]), "r"(r[o + 5]), "r"(r[o + 6]), "r"(r[o + 7])

__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : MFA_R8(r, 0), MFA_R8(r, 8), MFA_R8(r, 16), MFA_R8(r, 24)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : MFA_R8(r, 0), MFA_R8(r, 8)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_x32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%32], "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31};"
      ::MFA_W8(r, 0), MFA_W8(r, 8), MFA_W8(r, 16), MFA_W8(r, 24), "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%16], "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15};"
      ::MFA_W8(r, 0), MFA_W8(r, 8), "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_x8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%8], {%0, %1, %2, %3, %4, %5, %6, %7};" ::MFA_W8(r, 0), "r"(taddr)
               : "memory");
}

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// pack two fp32 into bf16x2 / f16x2: `lo` lands in bits [0,16), `hi` in [16,32)
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// two fp32 -> e4m3x2 (saturating): `lo` lands in bits [0,8), `hi` in [8,16)  (tools/f8_probe.cu: the first PTX operand is the high byte)
__device__ __forceinline__ uint32_t pack_e4m3(float lo, float hi) {
  unsigned short r;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(hi), "f"(lo));
  return (uint32_t)r;
}

// ---- packed fp32 pairs (sm_100 FFMA2 / FADD2): one issue slot for two lanes of softmax arithmetic
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) { f32x2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 add2_rm(f32x2 a, f32x2 b) { f32x2 r; asm("add.rm.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }

template <int N> __device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

}  // namespace ptx
}  // namespace mfa
