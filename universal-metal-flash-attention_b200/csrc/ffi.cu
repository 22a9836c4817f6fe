// ffi.cu -- the mfa_* C ABI (include/mfa_ffi.h, include/mfa_ffi_ext.h) over the CUDA kernels in this directory.
//
// Mirrors the behaviour of the reference's Swift bridge (Sources/MFABridge/MFABridge.swift,
// MFABridge+Quantized.swift) at the boundary: integer error codes, NULL handle -> 1, blocking compute calls with
// results visible in caller memory on return, a process-wide retained context singleton, strdup'd error strings.
// There is no CPU fallback anywhere: without an sm_100 device every compute entry point returns
// MFA_ERROR_DEVICE_NOT_SUPPORTED.
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/mfa_ffi_ext.h"
#include "common.h"
#include "tc_host.h"

using namespace mfa;

namespace mfa {
cudaError_t launch_quantize_grouped(const void* src, int src_dtype, void* codes, float* scales, uint64_t rows,
                                    uint64_t cols, uint32_t block_rows, uint32_t block_cols, uint64_t group_rows,
                                    int bits, float scale_floor, cudaStream_t st);
}

namespace {

bool g_debug = false;
#define DBG(...) do { if (g_debug) { fprintf(stderr, "[mfa] " __VA_ARGS__); fputc('\n', stderr); } } while (0)

// A call that the tensor-core kernels cannot serve runs on the exact fp32-math SIMT kernels, ~100x slower.  Small calls are
// served there by design; for anything sizeable say so ONCE per process and direction (MFA_QUIET_FALLBACK=1 silences it,
// last_kernel always tells the route).
void note_simt_route(const char* what, const AttnParams& p) {
  static bool said[2] = {false, false};
  const int i = what[0] == 'b' ? 1 : 0;
  if (said[i] || (double)p.B * p.H * p.Sq * p.Skv < 64.0 * 1024 * 1024 || getenv("MFA_QUIET_FALLBACK")) return;
  said[i] = true;
  const char* dt[] = {"fp16", "bf16", "fp32", "int8", "int4"};
  fprintf(stderr, "[mfa] %s of B=%d H=%d Sq=%d Skv=%d D=%d (%s operands) runs on the exact SIMT kernels, not the tensor pipe: "
          "tensor-core routes need a head_dim that is a multiple of 8 (<= 256 forward, <= 128 backward and fp32; int8 / int4: 128), unit stride along D, masks with unit key stride, "
          "no transposed operands\n", what, p.B, p.H, p.Sq, p.Skv, p.D, (p.in_dtype >= 0 && p.in_dtype <= 4) ? dt[p.in_dtype] : "?");
}

struct Scratch {
  void* ptr = nullptr;
  size_t cap = 0;
  // cross-stream ordering: the stream that used the block last and an event recorded behind that use (ScratchScope)
  cudaEvent_t ev = nullptr;
  cudaStream_t last = nullptr;
  bool used = false;
  // a captured CUDA graph holds the block's address: growing the block then retires it instead of freeing it, and retired blocks
  // are freed with the context, so a graph replayed later still writes memory it owns
  bool captured = false;
  std::vector<void*> retired;
  void* get(size_t bytes) {
    if (bytes <= cap) return ptr;
    if (ptr && captured) retired.push_back(ptr);
    else if (ptr) cudaFree(ptr);       // implicitly waits for everything that may still read the old block
    ptr = nullptr; cap = 0; used = false; captured = false;
    size_t want = bytes + (bytes >> 2) + 256;
    if (cudaMalloc(&ptr, want) != cudaSuccess) { ptr = nullptr; cudaGetLastError(); return nullptr; }
    cap = want;
    return ptr;
  }
  void release() {
    for (void* r : retired) cudaFree(r);
    retired.clear();
    captured = false;
    if (ptr) cudaFree(ptr);
    if (ev) cudaEventDestroy(ev);
    ptr = nullptr; cap = 0; ev = nullptr; used = false;
  }
};

struct Context {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // host-buffer pipeline (forward_pipelined): copy-in / copy-out streams and per-chunk events, created on first use
  cudaStream_t h2d = nullptr, d2h = nullptr;
  std::vector<cudaEvent_t> ev_in, ev_k0, ev_k1;
  double last_latency = 0.0;
  int refs = 0;
  std::recursive_mutex mu;          // recursive: mfa_quantized_backward holds it across quantise + backward_core
  enum { kMask, kLse, kDterm, kQCodes, kKCodes, kVCodes, kQScales, kKScales, kVScales, kTmpO, kQTmp, kMaskTiles, kKvSplit, kNumScratch };
  Scratch scratch[kNumScratch];
  std::vector<float> row_scales[3];
  const char* last_kernel = "none";
};

std::mutex g_ctx_mu;
constexpr int kMaxDevices = 64;
Context* g_ctxs[kMaxDevices] = {nullptr};   // one retained singleton per device (MFABridge.swift:652-687 keeps one per process:
                                            // a single-process host selects the device of the next create with mfa_set_device)
int g_device_request = -1;

int requested_device() {
  if (g_device_request >= 0) return g_device_request;
  if (const char* e = getenv("MFA_CUDA_DEVICE")) return atoi(e);
  return 0;
}

// Every entry point runs on its context's device and leaves the caller's current device as it found it.
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); }
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// Scratch blocks are shared by every call on a context.  Calls on different streams are ordered through an event recorded
// behind each use: a later call on another stream waits for it before touching the block (ADVICE r1: a blocking call could
// overwrite scratch an earlier async kernel was still reading).
struct ScratchScope {
  Context* ctx; cudaStream_t st;
  std::vector<int> slots;
  ScratchScope(Context* c, cudaStream_t s) : ctx(c), st(s) {}
  void* take(int slot, size_t bytes);
  ~ScratchScope();
};

void* ScratchScope::take(int slot, size_t bytes) {
  Scratch& sc = ctx->scratch[slot];
  void* p = sc.get(bytes);
  if (!p) return nullptr;
  // (a block a captured graph writes may be in use by a replay on any stream)
  if (sc.used && (sc.last != st || sc.captured) && sc.ev) cudaStreamWaitEvent(st, sc.ev, 0);
  slots.push_back(slot);
  return p;
}
ScratchScope::~ScratchScope() {
  for (int slot : slots) {
    Scratch& sc = ctx->scratch[slot];
    if (!sc.ev && cudaEventCreateWithFlags(&sc.ev, cudaEventDisableTiming) != cudaSuccess) { sc.ev = nullptr; cudaGetLastError(); continue; }
    cudaEventRecord(sc.ev, st);
    sc.last = st; sc.used = true;
  }
}

struct Buffer {
  Context* owner = nullptr;
  void* host = nullptr;   // CPU-dereferenceable pointer (may be null for pure device views)
  void* dev = nullptr;    // device pointer used by kernels
  size_t bytes = 0;
  bool owns_host = false, owns_dev = false, registered = false;
  bool mirrored = false;  // host and dev are distinct allocations kept coherent around compute calls
  int ndim = 0;
  int64_t shape[4] = {0, 0, 0, 0}, strides[4] = {0, 0, 0, 0};
};

bool device_ok(int dev) {
  static int cached[kMaxDevices];        // 0 unknown, 1 yes, 2 no
  static std::mutex mu;
  if (dev < 0 || dev >= kMaxDevices) return false;
  std::lock_guard<std::mutex> lock(mu);
  if (cached[dev]) return cached[dev] == 1;
  int n = 0, major = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || dev >= n ||
      cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) {
    cudaGetLastError();
    cached[dev] = 2;
    return false;
  }
  cached[dev] = (major == 10) ? 1 : 2;   // kernels are built for sm_100a only
  return cached[dev] == 1;
}
bool device_ok() { return device_ok(requested_device()); }

}  // namespace

namespace mfa {
// Watchdog builds (-DMFA_MBAR_WATCHDOG): a host-mapped buffer the kernels' mbarrier watchdog writes stuck waits into; it is
// ordinary pinned host memory, so it can still be read after the trap has killed the CUDA context.
struct WatchdogLogHost { unsigned int count; unsigned int pad; unsigned int rec[1024][4]; };
static WatchdogLogHost* g_wd_host = nullptr;
void* watchdog_device_log() {
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  if (!g_wd_host) {
    void* h = nullptr;
    if (cudaHostAlloc(&h, sizeof(WatchdogLogHost), cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    memset(h, 0, sizeof(WatchdogLogHost));
    g_wd_host = reinterpret_cast<WatchdogLogHost*>(h);
  }
  void* d = nullptr;
  if (cudaHostGetDevicePointer(&d, g_wd_host, 0) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return d;
}
static void watchdog_report() {
  if (!g_wd_host || g_wd_host->count == 0) return;
  const unsigned int n = g_wd_host->count < 1024 ? g_wd_host->count : 1024;
  fprintf(stderr, "[mfa] mbarrier watchdog: %u stuck wait(s); unique (block, warp, barrier smem address, parity) x threads:\n", g_wd_host->count);
  unsigned int shown = 0;
  for (unsigned int i = 0; i < n && shown < 256; ++i) {
    const unsigned int* r = g_wd_host->rec[i];
    bool dup = false;
    unsigned int same = 0;
    for (unsigned int j = 0; j < n; ++j) {
      const unsigned int* q = g_wd_host->rec[j];
      if (q[0] == r[0] && q[1] / 32 == r[1] / 32 && q[2] == r[2] && q[3] == r[3]) { if (j < i) dup = true; ++same; }
    }
    if (dup) continue;
    fprintf(stderr, "[mfa]   block %u warp %u bar 0x%x parity %u x%u\n", r[0], r[1] / 32, r[2], r[3], same);
    ++shown;
  }
  g_wd_host->count = 0;
}
}  // namespace mfa

namespace {

inline mfa_error_t cuda_fail(cudaError_t e, const char* what) {
  mfa::watchdog_report();
  DBG("%s: %s", what, cudaGetErrorString(e));
  cudaGetLastError();
  return e == cudaErrorMemoryAllocation ? MFA_ERROR_MEMORY_ALLOCATION : MFA_ERROR_EXECUTION_FAILED;
}

// --------------------------------------------------------------------------------------------------------------
// buffer <-> device coherence around a compute call
struct Sync {
  Context* ctx;
  cudaStream_t st;
  bool async;
  std::vector<Buffer*> outs;
  cudaError_t in(Buffer* b) {
    if (!b || !b->mirrored) return cudaSuccess;
    return cudaMemcpyAsync(b->dev, b->host, b->bytes, cudaMemcpyHostToDevice, st);
  }
  void out(Buffer* b) { if (b && b->mirrored) outs.push_back(b); }
  cudaError_t finish() {
    for (Buffer* b : outs) {
      cudaError_t e = cudaMemcpyAsync(b->host, b->dev, b->bytes, cudaMemcpyDeviceToHost, st);
      if (e != cudaSuccess) return e;
    }
    return async ? cudaSuccess : cudaStreamSynchronize(st);
  }
};

inline Buffer* B_(mfa_buffer_t h) { return reinterpret_cast<Buffer*>(h); }
inline Context* C_(mfa_context_t h) { return reinterpret_cast<Context*>(h); }

int parse_precision_str(const char* s) {   // MFABridge.swift:1438-1451: unknown -> fp32
  if (!s) return kF32;
  std::string v(s);
  for (auto& c : v) c = (char)tolower(c);
  if (v == "fp16" || v == "float16" || v == "half") return kF16;
  if (v == "bf16" || v == "bfloat16") return kBF16;
  if (v == "int8") return kI8;
  if (v == "int4") return kI4;
  return kF32;
}

TensorView contiguous_view(const void* p, int64_t H, int64_t S, int64_t D, bool transposed) {
  TensorView t;
  t.ptr = p;
  t.sb = H * S * D; t.sh = S * D;
  if (transposed) { t.ss = 1; t.sd = S; } else { t.ss = D; t.sd = 1; }
  return t;
}

// A buffer created *_with_strides carries BHSD element strides (last dim contiguous); otherwise contiguous.
TensorView view_of(Buffer* b, int64_t H, int64_t S, int64_t D, bool transposed) {
  TensorView t = contiguous_view(b->dev, H, S, D, transposed);
  if (b->ndim == 4 && !transposed) { t.sb = b->strides[0]; t.sh = b->strides[1]; t.ss = b->strides[2]; t.sd = b->strides[3]; }
  else if (b->ndim == 3 && !transposed) { t.sb = 0; t.sh = b->strides[0]; t.ss = b->strides[1]; t.sd = b->strides[2]; }
  return t;
}

// Does the handle cover a [B, H, S, D] operand of `esz`-byte elements?  Plain handles need B*H*S*D elements; handles made
// *_with_strides must carry exactly that shape (3-D handles: [H, S, D], batch 1) and their furthest element must lie inside.
bool view_fits(const Buffer* b, uint64_t B, uint64_t H, uint64_t S, uint64_t D, size_t esz) {
  if (!b) return false;
  if (b->ndim == 0) return b->bytes >= B * H * S * D * esz;
  const uint64_t want4[4] = {B, H, S, D};
  const uint64_t* want = b->ndim == 4 ? want4 : want4 + 1;
  if (b->ndim != 4 && b->ndim != 3) return false;
  if (b->ndim == 3 && B != 1) return false;
  uint64_t last = 0;
  for (int i = 0; i < b->ndim; ++i) {
    if (b->shape[i] != (int64_t)want[i] || b->strides[i] < 0) return false;
    if (want[i] == 0) return true;
    last += (want[i] - 1) * (uint64_t)b->strides[i];
  }
  return (last + 1) * esz <= b->bytes;
}

struct MaskArgs {
  const void* ptr; size_t bytes; const int64_t* shape; const int64_t* strides; uint32_t ndim; int type; int scalar;
};

// Resolve mask metadata into broadcast strides over [B,H,Sq,Skv] (right-aligned, size-1 dims broadcast:
// MFABridge.swift:186-198).  Host masks are copied into device scratch.  Returns 0 / error code.
mfa_error_t setup_mask(ScratchScope& scope, cudaStream_t st, const MaskArgs& m, AttnParams& p) {
  p.mask = nullptr; p.mask_kind = kMaskNone; p.mask_scalar = kMaskU8;
  p.mask_sb = p.mask_sh = p.mask_sq = p.mask_sk = 0;
  if (m.type == MFA_MASK_TYPE_NONE || !m.ptr || m.bytes == 0 || m.ndim == 0) return MFA_SUCCESS;
  if (!m.shape || m.ndim > 4) return MFA_ERROR_INVALID_ARGS;
  if (m.type != MFA_MASK_TYPE_BOOL && m.type != MFA_MASK_TYPE_ADDITIVE) return MFA_ERROR_INVALID_ARGS;
  if (m.type == MFA_MASK_TYPE_ADDITIVE && (m.scalar < MFA_MASK_SCALAR_FP16 || m.scalar > MFA_MASK_SCALAR_FP32))
    return MFA_ERROR_INVALID_ARGS;
  const int64_t full[4] = {p.B, p.H, p.Sq, p.Skv};
  int64_t bs[4] = {0, 0, 0, 0};
  int64_t contiguous = 1;
  std::vector<int64_t> cstr(m.ndim);
  for (int i = (int)m.ndim - 1; i >= 0; --i) { cstr[i] = contiguous; contiguous *= m.shape[i]; }
  const size_t esz = m.type == MFA_MASK_TYPE_BOOL ? 1 : (m.scalar == MFA_MASK_SCALAR_FP32 ? 4 : 2);
  int64_t max_index = 0;
  for (uint32_t i = 0; i < m.ndim; ++i) {
    int axis = 4 - (int)m.ndim + (int)i;
    int64_t dim = m.shape[i];
    if (dim != 1 && dim != full[axis]) return MFA_ERROR_INVALID_ARGS;
    int64_t s = m.strides ? m.strides[i] : cstr[i];
    bs[axis] = dim == 1 ? 0 : s;
    if (dim > 1) { if (s < 0) return MFA_ERROR_INVALID_ARGS; max_index += (dim - 1) * s; }
  }
  if ((size_t)(max_index + 1) * esz > m.bytes) return MFA_ERROR_INVALID_ARGS;
  cudaPointerAttributes attr;
  bool on_device = cudaPointerGetAttributes(&attr, m.ptr) == cudaSuccess &&
                   (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged);
  cudaGetLastError();
  const void* dptr = m.ptr;
  if (!on_device) {
    void* s = scope.take(Context::kMask, m.bytes);
    if (!s) return MFA_ERROR_MEMORY_ALLOCATION;
    if (cudaMemcpyAsync(s, m.ptr, m.bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) return MFA_ERROR_EXECUTION_FAILED;
    dptr = s;
  }
  p.mask = dptr;
  p.mask_kind = m.type == MFA_MASK_TYPE_BOOL ? kMaskBool : kMaskAdditive;
  p.mask_scalar = m.type == MFA_MASK_TYPE_BOOL ? kMaskU8 : m.scalar;
  p.mask_sb = bs[0]; p.mask_sh = bs[1]; p.mask_sq = bs[2]; p.mask_sk = bs[3];
  return MFA_SUCCESS;
}

size_t elems(uint32_t B, uint32_t H, uint32_t S, uint32_t D) { return (size_t)B * H * S * D; }

size_t packed_bytes(size_t n, int dtype) { return dtype == kI4 ? (n + 1) / 2 : n * dtype_bytes(dtype); }

void init_params(AttnParams& p, uint32_t B, uint32_t H, uint32_t Sq, uint32_t Skv, uint32_t D, float scale, bool causal,
                 int window) {
  memset(&p, 0, sizeof(p));
  p.B = (int)B; p.H = (int)H; p.Hkv = (int)H; p.Sq = (int)Sq; p.Skv = (int)Skv; p.D = (int)D;
  p.scale = scale; p.causal = causal ? 1 : 0; p.window = window;
  p.qq = p.qk = p.qv = QuantView{nullptr, 1.f, 0, 0};
  p.o_dtype = kF32; p.do_dtype = kF32;
}

// Packed variable-length sequences: the device offsets the kernels read (null buffers = dense).
void set_segments(AttnParams& p, const Buffer* cu_q, const Buffer* cu_k, uint32_t nseq) {
  if (!cu_q || !cu_k) return;
  p.cu_q = reinterpret_cast<const int*>(cu_q->dev);
  p.cu_k = reinterpret_cast<const int*>(cu_k->dev);
  p.nseq = (int)nseq;
}

// Arguments every varlen entry point checks before any device work: handles and num_seqs, then (with a device) sizes and --
// where the host can read them (host mirrors, managed memory) -- the offsets themselves: 0, non-decreasing, ending at the total.  Device-resident offsets are left to
// the kernels, which clamp every bound they derive from them (common.h).
mfa_error_t check_segments(const Buffer* cu_q, const Buffer* cu_k, uint32_t nseq, uint32_t total_q, uint32_t total_k) {
  if (!cu_q || !cu_k || nseq == 0 || nseq > 0x7ffffffeu) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  const size_t bytes = ((size_t)nseq + 1) * sizeof(int32_t);
  if (cu_q->bytes < bytes || cu_k->bytes < bytes || cu_q->ndim || cu_k->ndim) return MFA_ERROR_INVALID_ARGS;
  if (total_q > 0x7fffffffu || total_k > 0x7fffffffu) return MFA_ERROR_INVALID_ARGS;
  const struct { const Buffer* b; uint32_t total; } arrays[2] = {{cu_q, total_q}, {cu_k, total_k}};
  for (const auto& a : arrays) {
    if (!a.b->host) continue;
    const int32_t* cu = reinterpret_cast<const int32_t*>(a.b->host);
    if (cu[0] != 0 || cu[nseq] != (int64_t)a.total) return MFA_ERROR_INVALID_ARGS;
    for (uint32_t s = 0; s < nseq; ++s)
      if (cu[s + 1] < cu[s]) return MFA_ERROR_INVALID_ARGS;
  }
  return MFA_SUCCESS;
}

struct Timer {
  Context* ctx; cudaStream_t st; bool on;
  Timer(Context* c, cudaStream_t s, bool enable) : ctx(c), st(s), on(enable) { if (on) cudaEventRecord(ctx->ev0, st); }
  void stop() { if (on) cudaEventRecord(ctx->ev1, st); }
  void read() {
    if (!on) return;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_latency = ms * 1e-3;
    else cudaGetLastError();
  }
};

// ------------------------------------------------------------------------------------------ forward core
struct FwdArgs {
  Buffer *q, *k, *v, *out, *lse;
  uint32_t B, Sq, Skv, H, D;
  float scale; bool causal; int window;
  int in_dtype, out_dtype_req;
  bool tq, tk, tv, to;
  MaskArgs mask;
  cudaStream_t user_stream; bool async;
  // packed variable-length sequences (mfa_attention_forward_varlen): K / V heads (0 = H) and the segment offsets
  uint32_t Hkv;
  Buffer *cu_q, *cu_k; uint32_t nseq;
};

bool valid_float_dtype(int d) { return d == kF16 || d == kBF16 || d == kF32; }

// Host-buffer forward as a three-stage pipeline over (batch, head-group) chunks: H2D of chunk c+1, the attention
// kernel on chunk c and D2H of chunk c-1 overlap on separate streams (PCIe is full duplex), so the blocking call costs
// about max(H2D, D2H) instead of H2D + kernel + D2H.  (batch, head) units are independent (MultiHeadAttention.swift:
// 373-377), so each chunk is a complete attention problem on a contiguous slab of the caller's BHSD arrays.
// Used when Q, K, V and O are contiguous host mirrors and the tensor-core kernel applies; everything else takes the
// single-shot path below.
bool ensure_pipeline(Context* ctx, size_t chunks) {
  if (!ctx->h2d && cudaStreamCreateWithFlags(&ctx->h2d, cudaStreamNonBlocking) != cudaSuccess) return false;
  if (!ctx->d2h && cudaStreamCreateWithFlags(&ctx->d2h, cudaStreamNonBlocking) != cudaSuccess) return false;
  while (ctx->ev_in.size() < chunks) {
    cudaEvent_t a, b, c;
    if (cudaEventCreateWithFlags(&a, cudaEventDisableTiming) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess ||
        cudaEventCreate(&c) != cudaSuccess)
      return false;
    ctx->ev_in.push_back(a); ctx->ev_k0.push_back(b); ctx->ev_k1.push_back(c);
  }
  return true;
}

size_t pipeline_chunk_bytes() {
  static size_t v = 0;
  if (!v) { const char* e = getenv("MFA_PIPELINE_CHUNK_MB"); v = (size_t)((e ? atof(e) : 16.0) * 1048576.0); if (!v) v = 1; }
  return v;
}

bool forward_pipeline_ok(const FwdArgs& a, int o_dtype) {
  if (a.async || a.cu_q || getenv("MFA_DISABLE_PIPELINE")) return false;
  if (!a.q->mirrored || !a.k->mirrored || !a.v->mirrored || !a.out->mirrored || (a.lse && !a.lse->mirrored)) return false;
  if (a.q->ndim || a.k->ndim || a.v->ndim || a.out->ndim) return false;
  if (a.tq || a.tk || a.tv || a.to) return false;
  if (a.mask.type != MFA_MASK_TYPE_NONE && a.mask.ptr && a.mask.bytes) return false;
  if (a.in_dtype != kBF16 && a.in_dtype != kF16) return false;
  if (a.D != 64 && a.D != 128 && a.D != 256) return false;
  (void)o_dtype;
  const size_t per_head = ((size_t)a.Sq + 2 * (size_t)a.Skv) * a.D * 2;
  return (size_t)a.B * a.H * per_head >= 2 * pipeline_chunk_bytes();     // small problems: one shot is as fast
}

mfa_error_t forward_pipelined(Context* ctx, const FwdArgs& a, int o_dtype) {
  const size_t esz = 2, oes = dtype_bytes(o_dtype);
  const size_t q_head = (size_t)a.Sq * a.D, kv_head = (size_t)a.Skv * a.D;
  const size_t per_head = (q_head + 2 * kv_head) * esz;
  uint32_t hc = (uint32_t)std::max<size_t>(1, (pipeline_chunk_bytes() + per_head / 2) / per_head);
  if (hc > a.H) hc = a.H;
  const uint32_t groups = (a.H + hc - 1) / hc;
  const size_t chunks = (size_t)a.B * groups;
  if (!ensure_pipeline(ctx, chunks)) return MFA_ERROR_MEMORY_ALLOCATION;
  cudaStream_t st = ctx->stream;
  cudaError_t e = cudaSuccess;
  size_t c = 0;
  auto at = [](void* base, size_t off) { return reinterpret_cast<uint8_t*>(base) + off; };
  for (uint32_t b = 0; b < a.B && e == cudaSuccess; ++b) {
    for (uint32_t g = 0; g < groups && e == cudaSuccess; ++g, ++c) {
      const uint32_t h0 = g * hc, hn = std::min(hc, a.H - h0);
      const size_t qo = ((size_t)b * a.H + h0) * q_head, ko = ((size_t)b * a.H + h0) * kv_head;
      if ((e = cudaMemcpyAsync(at(a.q->dev, qo * esz), at(a.q->host, qo * esz), hn * q_head * esz, cudaMemcpyHostToDevice, ctx->h2d)) != cudaSuccess) break;
      if ((e = cudaMemcpyAsync(at(a.k->dev, ko * esz), at(a.k->host, ko * esz), hn * kv_head * esz, cudaMemcpyHostToDevice, ctx->h2d)) != cudaSuccess) break;
      if ((e = cudaMemcpyAsync(at(a.v->dev, ko * esz), at(a.v->host, ko * esz), hn * kv_head * esz, cudaMemcpyHostToDevice, ctx->h2d)) != cudaSuccess) break;
      cudaEventRecord(ctx->ev_in[c], ctx->h2d);
      cudaStreamWaitEvent(st, ctx->ev_in[c], 0);
      AttnParams p;
      init_params(p, 1, hn, a.Sq, a.Skv, a.D, a.scale, a.causal, a.window);
      p.q = contiguous_view(at(a.q->dev, qo * esz), hn, a.Sq, a.D, false);
      p.k = contiguous_view(at(a.k->dev, ko * esz), hn, a.Skv, a.D, false);
      p.v = contiguous_view(at(a.v->dev, ko * esz), hn, a.Skv, a.D, false);
      p.o = contiguous_view(at(a.out->dev, qo * oes), hn, a.Sq, a.D, false);
      const size_t lo = ((size_t)b * a.H + h0) * a.Sq;
      p.lse = a.lse ? reinterpret_cast<float*>(a.lse->dev) + lo : nullptr;
      p.in_dtype = a.in_dtype; p.o_dtype = o_dtype;
      if (!fwd_tc_eligible(p)) { e = cudaErrorNotSupported; break; }
      cudaEventRecord(ctx->ev_k0[c], st);
      if ((e = launch_fwd_tc(p, st)) != cudaSuccess) break;
      cudaEventRecord(ctx->ev_k1[c], st);
      cudaStreamWaitEvent(ctx->d2h, ctx->ev_k1[c], 0);
      if ((e = cudaMemcpyAsync(at(a.out->host, qo * oes), at(a.out->dev, qo * oes), hn * q_head * oes, cudaMemcpyDeviceToHost, ctx->d2h)) != cudaSuccess) break;
      if (a.lse) e = cudaMemcpyAsync(at(a.lse->host, lo * 4), at(a.lse->dev, lo * 4), (size_t)hn * a.Sq * 4, cudaMemcpyDeviceToHost, ctx->d2h);
    }
  }
  cudaError_t e1 = cudaStreamSynchronize(ctx->d2h), e2 = cudaStreamSynchronize(st), e3 = cudaStreamSynchronize(ctx->h2d);
  ctx->last_kernel = g_last_kernel;
  if (e != cudaSuccess) return cuda_fail(e, "pipelined forward");
  if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) return cuda_fail(e1 != cudaSuccess ? e1 : e2 != cudaSuccess ? e2 : e3, "pipelined forward sync");
  double total = 0.0;                      // mfa_get_gpu_latency: kernel time only, summed over the chunks
  for (size_t i = 0; i < chunks; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev_k0[i], ctx->ev_k1[i]) == cudaSuccess) total += ms * 1e-3; else cudaGetLastError();
  }
  ctx->last_latency = total;
  return MFA_SUCCESS;
}

mfa_error_t forward_core(Context* ctx, const FwdArgs& a) {
  if (!ctx || !a.q || !a.k || !a.v || !a.out) return MFA_ERROR_INVALID_ARGS;
  if (!valid_float_dtype(a.in_dtype)) return MFA_ERROR_INVALID_ARGS;
  if (a.D == 0 || a.D > 256 || a.H == 0) return MFA_ERROR_INVALID_ARGS;
  const uint32_t Hkv = a.Hkv ? a.Hkv : a.H;
  if (a.H % Hkv) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  const size_t nq = elems(a.B, a.H, a.Sq, a.D), nkv = elems(a.B, Hkv, a.Skv, a.D);
  const size_t esz = dtype_bytes(a.in_dtype);
  if (!view_fits(a.q, a.B, a.H, a.Sq, a.D, esz) || !view_fits(a.k, a.B, Hkv, a.Skv, a.D, esz) ||
      !view_fits(a.v, a.B, Hkv, a.Skv, a.D, esz))
    return MFA_ERROR_INVALID_ARGS;
  // O is fp32 (reference contract) unless the handle only fits the requested lower precision.
  int o_dtype = kF32;
  if (a.out->bytes < nq * 4) {
    if (valid_float_dtype(a.out_dtype_req) && a.out->bytes >= nq * dtype_bytes(a.out_dtype_req)) o_dtype = a.out_dtype_req;
    else return MFA_ERROR_INVALID_ARGS;
  }
  if (a.lse && a.lse->bytes < (size_t)a.B * a.H * a.Sq * 4) return MFA_ERROR_INVALID_ARGS;
  if (a.async && (a.q->mirrored || a.k->mirrored || a.v->mirrored || a.out->mirrored || (a.lse && a.lse->mirrored) ||
                  (a.cu_q && (a.cu_q->mirrored || a.cu_k->mirrored))))
    return MFA_ERROR_INVALID_ARGS;

  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  if (nq != 0 && nkv != 0 && forward_pipeline_ok(a, o_dtype)) {
    // the pipeline only drives the tensor-core kernel: probe eligibility on one head's worth of the problem first and take
    // the single-shot path (which may route to the exact SIMT kernel) when it does not apply
    AttnParams probe;
    init_params(probe, 1, 1, a.Sq, a.Skv, a.D, a.scale, a.causal, a.window);
    probe.q = contiguous_view(a.q->dev, 1, a.Sq, a.D, false);
    probe.k = contiguous_view(a.k->dev, 1, a.Skv, a.D, false);
    probe.v = contiguous_view(a.v->dev, 1, a.Skv, a.D, false);
    probe.o = contiguous_view(a.out->dev, 1, a.Sq, a.D, false);
    probe.in_dtype = a.in_dtype; probe.o_dtype = o_dtype;
    if (fwd_tc_eligible(probe)) return forward_pipelined(ctx, a, o_dtype);
  }
  cudaStream_t st = a.async ? a.user_stream : ctx->stream;
  ScratchScope scope(ctx, st);
  Sync sync{ctx, st, a.async, {}};
  cudaError_t e;
  if ((e = sync.in(a.q)) != cudaSuccess || (e = sync.in(a.k)) != cudaSuccess || (e = sync.in(a.v)) != cudaSuccess ||
      (e = sync.in(a.cu_q)) != cudaSuccess || (e = sync.in(a.cu_k)) != cudaSuccess)
    return cuda_fail(e, "h2d");
  if (nq == 0) { return sync.finish() == cudaSuccess ? MFA_SUCCESS : MFA_ERROR_EXECUTION_FAILED; }

  AttnParams p;
  init_params(p, a.B, a.H, a.Sq, a.Skv, a.D, a.scale, a.causal, a.window);
  p.Hkv = (int)Hkv;
  p.q = view_of(a.q, a.H, a.Sq, a.D, a.tq);
  p.k = view_of(a.k, Hkv, a.Skv, a.D, a.tk);
  p.v = view_of(a.v, Hkv, a.Skv, a.D, a.tv);
  p.o = view_of(a.out, a.H, a.Sq, a.D, a.to);
  p.lse = a.lse ? reinterpret_cast<float*>(a.lse->dev) : nullptr;
  p.in_dtype = a.in_dtype; p.o_dtype = o_dtype;
  set_segments(p, a.cu_q, a.cu_k, a.nseq);
  mfa_error_t me = setup_mask(scope, st, a.mask, p);
  if (me != MFA_SUCCESS) return me;

  if (const size_t mb = fwd_tc_mask_scratch_bytes(p))
    p.mask_tile_scratch = reinterpret_cast<int*>(scope.take(Context::kMaskTiles, mb));     // null = no tile skipping
  Timer tm(ctx, st, !a.async);
  if (fwd_tc_eligible(p)) {
    e = launch_fwd_tc(p, st);
  } else if (fwd_split_eligible(p)) {
    // fp32 operands (the reference adapters' default precision) at head_dim 128: tensor pipe through fp16 (hi, lo) pairs
    void* tmp = scope.take(Context::kQTmp, fwd_split_scratch_bytes(p));
    if (!tmp) return MFA_ERROR_MEMORY_ALLOCATION;
    e = launch_fwd_split(p, tmp, st);
  } else {
    note_simt_route("forward", p);
    e = launch_fwd_simt(p, st);
  }
  tm.stop();
  ctx->last_kernel = g_last_kernel;
  if (e != cudaSuccess) return cuda_fail(e, "forward launch");
  sync.out(a.out); sync.out(a.lse);
  if ((e = sync.finish()) != cudaSuccess) return cuda_fail(e, "forward sync");
  tm.read();
  return MFA_SUCCESS;
}

// ------------------------------------------------------------------------------------------ backward core
struct BwdArgs {
  Buffer *dout, *q, *k, *v, *out, *lse, *dq, *dk, *dv, *dbuf;
  uint32_t B, Sq, Skv, H, Hkv, D;
  float scale; bool causal; int window;
  int in_dtype, do_dtype;
  bool tq, tk, tv, to;
  MaskArgs mask;
  QuantView qq, qk, qv;
  cudaStream_t user_stream; bool async;
  bool want_dq, want_dkv;
  Buffer *cu_q, *cu_k; uint32_t nseq;         // packed variable-length sequences (mfa_attention_backward_varlen)
};

mfa_error_t backward_core(Context* ctx, const BwdArgs& a) {
  if (!ctx || !a.dout || !a.q || !a.k || !a.v || !a.out || !a.lse) return MFA_ERROR_INVALID_ARGS;
  if ((a.want_dq && !a.dq) || (a.want_dkv && (!a.dk || !a.dv))) return MFA_ERROR_INVALID_ARGS;
  if (a.D == 0 || a.D > 256 || a.H == 0 || a.Hkv == 0 || a.H % a.Hkv) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  const size_t nq = elems(a.B, a.H, a.Sq, a.D), nkv = elems(a.B, a.Hkv, a.Skv, a.D);
  const size_t rows = (size_t)a.B * a.H * a.Sq;
  if (a.q->bytes < packed_bytes(nq, a.in_dtype) || a.k->bytes < packed_bytes(nkv, a.in_dtype) ||
      a.v->bytes < packed_bytes(nkv, a.in_dtype))
    return MFA_ERROR_INVALID_ARGS;
  if (a.dout->bytes < nq * dtype_bytes(a.do_dtype) || a.out->bytes < nq * 4 || a.lse->bytes < rows * 4)
    return MFA_ERROR_INVALID_ARGS;
  if ((a.want_dq && a.dq->bytes < nq * 4) || (a.want_dkv && (a.dk->bytes < nkv * 4 || a.dv->bytes < nkv * 4)))
    return MFA_ERROR_INVALID_ARGS;
  if (a.dbuf && a.dbuf->bytes < rows * 4) return MFA_ERROR_INVALID_ARGS;

  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  cudaStream_t st = a.async ? a.user_stream : ctx->stream;
  ScratchScope scope(ctx, st);
  Sync sync{ctx, st, a.async, {}};
  Buffer* ins[] = {a.dout, a.q, a.k, a.v, a.out, a.lse, a.cu_q, a.cu_k};
  for (Buffer* b : ins) {
    if (!b) continue;
    if (a.async && b->mirrored) return MFA_ERROR_INVALID_ARGS;
    cudaError_t e = sync.in(b);
    if (e != cudaSuccess) return cuda_fail(e, "h2d");
  }
  if (nq == 0 && nkv == 0) return MFA_SUCCESS;

  AttnParams p;
  init_params(p, a.B, a.H, a.Sq, a.Skv, a.D, a.scale, a.causal, a.window);
  p.Hkv = (int)a.Hkv;
  p.q = view_of(a.q, a.H, a.Sq, a.D, a.tq);
  p.k = view_of(a.k, a.Hkv, a.Skv, a.D, a.tk);
  p.v = view_of(a.v, a.Hkv, a.Skv, a.D, a.tv);
  p.o = contiguous_view(a.out->dev, a.H, a.Sq, a.D, a.to);
  p.d_o = contiguous_view(a.dout->dev, a.H, a.Sq, a.D, a.to);
  p.lse = reinterpret_cast<float*>(a.lse->dev);
  p.in_dtype = a.in_dtype; p.o_dtype = kF32; p.do_dtype = a.do_dtype;
  p.qq = a.qq; p.qk = a.qk; p.qv = a.qv;
  set_segments(p, a.cu_q, a.cu_k, a.nseq);
  p.dq = a.want_dq ? reinterpret_cast<float*>(a.dq->dev) : nullptr;
  p.dk = a.want_dkv ? reinterpret_cast<float*>(a.dk->dev) : nullptr;
  p.dv = a.want_dkv ? reinterpret_cast<float*>(a.dv->dev) : nullptr;
  if (a.dbuf) p.dterm = reinterpret_cast<float*>(a.dbuf->dev);
  else {
    p.dterm = reinterpret_cast<float*>(scope.take(Context::kDterm, rows * 4 + 4));
    if (!p.dterm) return MFA_ERROR_MEMORY_ALLOCATION;
  }
  mfa_error_t me = setup_mask(scope, st, a.mask, p);
  if (me != MFA_SUCCESS) return me;

  if (const size_t mb = bwd_tc_mask_scratch_bytes(p))
    p.mask_tile_scratch = reinterpret_cast<int*>(scope.take(Context::kMaskTiles, mb));     // null = no tile skipping
  Timer tm(ctx, st, !a.async);
  cudaError_t e = cudaSuccess;
  // Quantised operands at the head dim the quantised tensor-core forward serves (128): the backward runs on the tensor pipe
  // too, over the values the reference's backward sees (dequantised codes: QuantizedAttention.swift:1428-1608,
  // MFABridge+Quantized.swift:365-533) held as bf16 -- one HBM-bound pass per operand, then the bf16 dK/dV and dQ kernels.
  // Other head dims keep the exact SIMT route (dequantise on load).
  const char* tcq_name = nullptr;
  if ((p.in_dtype == kI8 || p.in_dtype == kI4) && a.D == 128 && !a.tq && !a.tk && !a.tv && !a.to &&
      !getenv("MFA_DISABLE_TC")) {
    auto packed_ok = [&](const TensorView& t, int64_t Hn, int64_t S) {
      return t.sd == 1 && t.ss == (int64_t)a.D && t.sh == S * (int64_t)a.D && t.sb == Hn * S * (int64_t)a.D;
    };
    if (packed_ok(p.q, a.H, a.Sq) && packed_ok(p.k, a.Hkv, a.Skv) && packed_ok(p.v, a.Hkv, a.Skv)) {
      const size_t qb = (nq * 2 + 255) & ~(size_t)255, kb = (nkv * 2 + 255) & ~(size_t)255;
      uint8_t* tmp = reinterpret_cast<uint8_t*>(scope.take(Context::kQTmp, 2 * qb + 2 * kb + 256));
      if (!tmp) return MFA_ERROR_MEMORY_ALLOCATION;
      const int bits = p.in_dtype == kI8 ? 8 : 4;
      void *q16 = tmp, *k16 = tmp + qb, *v16 = tmp + qb + kb, *g16 = tmp + qb + 2 * kb;
      e = launch_dequantize_bf16(p.q.ptr, bits, p.qq, q16, (uint64_t)a.B * a.H, a.Sq, a.D, st);
      if (e == cudaSuccess) e = launch_dequantize_bf16(p.k.ptr, bits, p.qk, k16, (uint64_t)a.B * a.Hkv, a.Skv, a.D, st);
      if (e == cudaSuccess) e = launch_dequantize_bf16(p.v.ptr, bits, p.qv, v16, (uint64_t)a.B * a.Hkv, a.Skv, a.D, st);
      const void* g = a.dout->dev;
      if (e == cudaSuccess && a.do_dtype != kBF16) { e = launch_to_bf16(g, a.do_dtype, g16, nq, st); g = g16; }
      if (e != cudaSuccess) return cuda_fail(e, "dequantise for the tensor-core backward");
      tcq_name = p.in_dtype == kI8 ? "bwd_tcq_int8_d128" : "bwd_tcq_int4_d128";
      p.q = contiguous_view(q16, a.H, a.Sq, a.D, false);
      p.k = contiguous_view(k16, a.Hkv, a.Skv, a.D, false);
      p.v = contiguous_view(v16, a.Hkv, a.Skv, a.D, false);
      p.d_o = contiguous_view(g, a.H, a.Sq, a.D, false);
      p.in_dtype = kBF16; p.do_dtype = kBF16;
      p.qq = p.qk = p.qv = QuantView{nullptr, 1.f, 0, 0};
    }
  }
  if (bwd_tc_eligible(p)) {
    e = launch_dterm(p, st);
    if (e == cudaSuccess) e = launch_bwd_tc(p, st);
    if (e == cudaSuccess && tcq_name) g_last_kernel = tcq_name;
  } else {
    note_simt_route("backward", p);
    e = launch_bwd_simt(p, st);   // empty Sq / Skv degrade to zero-filled gradients inside the kernels
  }
  tm.stop();
  ctx->last_kernel = g_last_kernel;
  if (e != cudaSuccess) return cuda_fail(e, "backward launch");
  if (a.want_dq) sync.out(a.dq);
  if (a.want_dkv) { sync.out(a.dk); sync.out(a.dv); }
  sync.out(a.dbuf);
  if ((e = sync.finish()) != cudaSuccess) return cuda_fail(e, "backward sync");
  tm.read();
  return MFA_SUCCESS;
}

// ------------------------------------------------------------------------------- quantised forward core
// Each operand is either floating point (quantised here to `target_bits` with `block_rows`-token blocks, 0 =
// per tensor) or already int8/int4 codes with a per-tensor scale / zero point (or per-row scales from
// mfa_set_scale_arrays).  Attention then runs on the dequantised values (reference semantics,
// QuantizedAttention.swift:71-91); lse optional.
struct QOperand { Buffer* buf; int dtype; float scale; int zp; uint32_t block_rows; };

struct QFwdArgs {
  QOperand q, k, v;
  Buffer *out, *lse, *mask_buf;
  uint32_t B, Sq, Skv, H, D;
  float scale; bool causal;
  int target_dtype;      // kI8 / kI4 for runtime-quantised float operands
  int out_dtype_req;
  bool use_row_scales;
};

mfa_error_t quantise_operand(ScratchScope& scope, cudaStream_t st, const QOperand& op, int which, uint32_t B, uint32_t H,
                             uint32_t S, uint32_t D, int target_dtype, TensorView& view, QuantView& qv, int& dtype_out) {
  const size_t n = elems(B, H, S, D);
  if (op.dtype == kI8 || op.dtype == kI4) {
    if (op.buf->bytes < packed_bytes(n, op.dtype)) return MFA_ERROR_INVALID_ARGS;
    view = contiguous_view(op.buf->dev, H, S, D, false);
    qv = QuantView{nullptr, op.scale, op.zp, 0};
    dtype_out = op.dtype;
    return MFA_SUCCESS;
  }
  if (!valid_float_dtype(op.dtype)) return MFA_ERROR_INVALID_ARGS;
  if (op.buf->bytes < n * dtype_bytes(op.dtype)) return MFA_ERROR_INVALID_ARGS;
  if (target_dtype != kI8 && target_dtype != kI4) {   // nothing asks for integers: keep floating point
    view = contiguous_view(op.buf->dev, H, S, D, false);
    qv = QuantView{nullptr, 1.f, 0, 0};
    dtype_out = op.dtype;
    return MFA_SUCCESS;
  }
  const int bits = target_dtype == kI8 ? 8 : 4;
  const uint64_t rows = (uint64_t)B * H * S;
  const uint32_t br = op.block_rows;                          // 0 = per tensor
  const uint64_t nb = br ? (uint64_t)B * H * ((S + br - 1) / br) : 1;
  void* codes = scope.take(Context::kQCodes + which, packed_bytes(n, target_dtype) + 16);
  float* scales = reinterpret_cast<float*>(scope.take(Context::kQScales + which, nb * 4 + 16));
  if (!codes || !scales) return MFA_ERROR_MEMORY_ALLOCATION;
  cudaError_t e = launch_quantize_grouped(op.buf->dev, op.dtype, codes, scales, rows, D, br ? br : (uint32_t)0, D,
                                          br ? S : 0, bits, 1e-8f, st);
  if (e != cudaSuccess) return cuda_fail(e, "quantise");
  view = contiguous_view(codes, H, S, D, false);
  qv = QuantView{scales, 1.f, 0, (int)br};
  dtype_out = target_dtype;
  return MFA_SUCCESS;
}

}  // namespace

// The quantised kernels take one in_dtype for Q, K and V; mixed operands are normalised by the callers below.
namespace {

mfa_error_t qforward_core(Context* ctx, const QFwdArgs& a) {
  if (!ctx || !a.q.buf || !a.k.buf || !a.v.buf || !a.out) return MFA_ERROR_INVALID_ARGS;
  if (a.D == 0 || a.D > 256 || a.H == 0) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  const size_t nq = elems(a.B, a.H, a.Sq, a.D);
  int o_dtype = kF32;
  if (a.out->bytes < nq * 4) {
    if (valid_float_dtype(a.out_dtype_req) && a.out->bytes >= nq * dtype_bytes(a.out_dtype_req)) o_dtype = a.out_dtype_req;
    else return MFA_ERROR_INVALID_ARGS;
  }
  if (a.lse && a.lse->bytes < (size_t)a.B * a.H * a.Sq * 4) return MFA_ERROR_INVALID_ARGS;
  if (a.mask_buf && a.mask_buf->bytes < (size_t)a.B * a.H * a.Sq * a.Skv * 4) return MFA_ERROR_INVALID_ARGS;

  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  cudaStream_t st = ctx->stream;
  ScratchScope scope(ctx, st);
  Sync sync{ctx, st, false, {}};
  cudaError_t e;
  if ((e = sync.in(a.q.buf)) != cudaSuccess || (e = sync.in(a.k.buf)) != cudaSuccess ||
      (e = sync.in(a.v.buf)) != cudaSuccess || (e = sync.in(a.mask_buf)) != cudaSuccess)
    return cuda_fail(e, "h2d");
  if (nq == 0) return MFA_SUCCESS;

  AttnParams p;
  init_params(p, a.B, a.H, a.Sq, a.Skv, a.D, a.scale, a.causal, -1);
  Timer tm(ctx, st, true);
  int dq_, dk_, dv_;
  mfa_error_t me;
  if ((me = quantise_operand(scope, st, a.q, 0, a.B, a.H, a.Sq, a.D, a.target_dtype, p.q, p.qq, dq_)) != MFA_SUCCESS) return me;
  if ((me = quantise_operand(scope, st, a.k, 1, a.B, a.H, a.Skv, a.D, a.target_dtype, p.k, p.qk, dk_)) != MFA_SUCCESS) return me;
  if ((me = quantise_operand(scope, st, a.v, 2, a.B, a.H, a.Skv, a.D, a.target_dtype, p.v, p.qv, dv_)) != MFA_SUCCESS) return me;
  if (dq_ != dk_ || dk_ != dv_) return MFA_ERROR_INVALID_ARGS;   // callers normalise mixed operands first
  p.in_dtype = dq_;
  if (a.use_row_scales && (dq_ == kI8 || dq_ == kI4)) {
    // per-row scales handed over through mfa_set_scale_arrays for pre-quantised operands
    const size_t want[3] = {(size_t)a.B * a.H * a.Sq, (size_t)a.B * a.H * a.Skv, (size_t)a.B * a.H * a.Skv};
    QuantView* qv[3] = {&p.qq, &p.qk, &p.qv};
    const QOperand* ops[3] = {&a.q, &a.k, &a.v};
    for (int i = 0; i < 3; ++i) {
      if ((ops[i]->dtype == kI8 || ops[i]->dtype == kI4) && ctx->row_scales[i].size() == want[i]) {
        float* s = reinterpret_cast<float*>(scope.take(Context::kQScales + i, want[i] * 4));
        if (!s) return MFA_ERROR_MEMORY_ALLOCATION;
        if ((e = cudaMemcpyAsync(s, ctx->row_scales[i].data(), want[i] * 4, cudaMemcpyHostToDevice, st)) != cudaSuccess)
          return cuda_fail(e, "row scales");
        *qv[i] = QuantView{s, 1.f, ops[i]->zp, 1};
      }
    }
  }
  p.o = contiguous_view(a.out->dev, a.H, a.Sq, a.D, false);
  p.o_dtype = o_dtype;
  p.lse = a.lse ? reinterpret_cast<float*>(a.lse->dev) : nullptr;
  if (a.mask_buf) {
    p.mask = a.mask_buf->dev; p.mask_kind = kMaskAdditive; p.mask_scalar = kMaskF32;
    p.mask_sk = 1; p.mask_sq = a.Skv; p.mask_sh = (int64_t)a.Sq * a.Skv; p.mask_sb = (int64_t)a.H * a.Sq * a.Skv;
  }
  if (const size_t mb = fwd_tc_mask_scratch_bytes(p))
    p.mask_tile_scratch = reinterpret_cast<int*>(scope.take(Context::kMaskTiles, mb));
  if (fwd_tcq_eligible(p)) {
    void* tmp = scope.take(Context::kQTmp, fwd_tcq_scratch_bytes(p));
    if (!tmp) return MFA_ERROR_MEMORY_ALLOCATION;
    e = launch_fwd_tcq(p, tmp, st);
  } else {
    note_simt_route("forward", p);
    e = launch_fwd_simt(p, st);
  }
  tm.stop();
  ctx->last_kernel = g_last_kernel;
  if (e != cudaSuccess) return cuda_fail(e, "quantised forward launch");
  sync.out(a.out); sync.out(a.lse);
  if ((e = sync.finish()) != cudaSuccess) return cuda_fail(e, "quantised forward sync");
  tm.read();
  return MFA_SUCCESS;
}

mfa_error_t make_buffer(Context* ctx, void* ptr, size_t bytes, bool device_hint, const int64_t* shape,
                        const int64_t* strides, uint32_t ndim, mfa_buffer_t* out) {
  if (!ctx || !out || !ptr) return MFA_ERROR_INVALID_ARGS;
  if (ndim > 4 || (ndim && (!shape || !strides))) return MFA_ERROR_INVALID_ARGS;
  Buffer* b = new (std::nothrow) Buffer();
  if (!b) return MFA_ERROR_MEMORY_ALLOCATION;
  b->owner = ctx;
  b->bytes = bytes;
  b->ndim = (int)ndim;
  for (uint32_t i = 0; i < ndim; ++i) { b->shape[i] = shape[i]; b->strides[i] = strides[i]; }
  bool on_device = device_hint;
  bool managed = false;
  DeviceGuard dg(ctx->device);
  if (device_ok(ctx->device)) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, ptr) == cudaSuccess) {
      if (attr.type == cudaMemoryTypeDevice) on_device = true;
      else if (attr.type == cudaMemoryTypeManaged) { on_device = true; managed = true; }
      else if (attr.type == cudaMemoryTypeHost && !device_hint) {
        // pinned host memory: mirror it (kernels reading host memory over PCIe would be far slower than a copy)
        on_device = false;
      }
    }
    cudaGetLastError();
  }
  if (on_device) {
    b->dev = ptr;
    b->host = managed ? ptr : nullptr;
  } else {
    b->host = ptr;
    b->mirrored = true;
    if (device_ok(ctx->device) && bytes) {
      if (cudaMalloc(&b->dev, bytes) != cudaSuccess) { cudaGetLastError(); delete b; return MFA_ERROR_MEMORY_ALLOCATION; }
      cudaMemset(b->dev, 0, bytes);       // an output mirror is copied back whole: bytes a kernel never wrote must not be garbage
      b->owns_dev = true;
      // Pin the caller's pages so the per-call copies run at full PCIe rate; failure is harmless.
      if (bytes >= (1u << 16) && cudaHostRegister(ptr, bytes, cudaHostRegisterDefault) == cudaSuccess) b->registered = true;
      cudaGetLastError();
    }
  }
  *out = b;
  return MFA_SUCCESS;
}

const char* kErrStr[] = {"Success", "Invalid arguments", "Memory allocation failed", "Device not supported",
                         "Kernel compilation failed", "Execution failed"};

int header_precision_to_dtype(int p) { return (p >= 0 && p <= 4) ? p : -1; }

}  // namespace

// ================================================================================================ C ABI
extern "C" {

void mfa_get_quantized_layout(mfa_quantized_kernel_t, mfa_quantized_layout_t* out_layout) {
  if (!out_layout) return;
  int32_t* f = reinterpret_cast<int32_t*>(out_layout);
  for (size_t i = 0; i < sizeof(mfa_quantized_layout_t) / sizeof(int32_t); ++i) f[i] = -1;
}

void mfa_get_quantized_capabilities(void* out_capabilities) {
  if (!out_capabilities) return;
  mfa_quantized_capabilities_t c;
  memset(&c, 0, sizeof(c));
  c.supports_multi_head_backward = true;
  c.supports_blockwise_backward = true;
  c.max_heads = 65535;
  c.max_block_size = 1024;
  memcpy(out_capabilities, &c, sizeof(c));
}

mfa_error_t mfa_set_device(int32_t device_index) {
  // Selects the device of the contexts created from now on.  Every device has its own retained context, so a single-process
  // host drives several GPUs by alternating mfa_set_device(i) / mfa_create_context (heads or batches sharded over the contexts).
  if (device_index < 0 || device_index >= kMaxDevices) return MFA_ERROR_INVALID_ARGS;
  int n = 0;
  if (cudaGetDeviceCount(&n) == cudaSuccess && n > 0 && device_index >= n) return MFA_ERROR_INVALID_ARGS;
  cudaGetLastError();
  std::lock_guard<std::mutex> lock(g_ctx_mu);
  g_device_request = device_index;
  return MFA_SUCCESS;
}

int32_t mfa_get_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

mfa_error_t mfa_create_context(mfa_context_t* context) {
  if (!context) return MFA_ERROR_INVALID_ARGS;
  *context = nullptr;
  if (const char* d = getenv("MFA_DEBUG")) g_debug = d[0] && d[0] != '0';
  std::lock_guard<std::mutex> lock(g_ctx_mu);
  const int dev = requested_device();
  if (dev < 0 || dev >= kMaxDevices) return MFA_ERROR_INVALID_ARGS;
  if (!g_ctxs[dev]) {
    if (!device_ok(dev)) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
    Context* c = new (std::nothrow) Context();
    if (!c) return MFA_ERROR_MEMORY_ALLOCATION;
    c->device = dev;
    DeviceGuard dg(dev);
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) {
      cudaGetLastError();
      delete c;
      return MFA_ERROR_DEVICE_NOT_SUPPORTED;
    }
    g_ctxs[dev] = c;
  }
  ++g_ctxs[dev]->refs;
  *context = g_ctxs[dev];
  return MFA_SUCCESS;
}

void mfa_destroy_context(mfa_context_t context) {
  if (!context) return;
  std::lock_guard<std::mutex> lock(g_ctx_mu);
  Context* c = nullptr;
  for (int i = 0; i < kMaxDevices; ++i) if (g_ctxs[i] && g_ctxs[i] == context) { c = g_ctxs[i]; break; }
  if (!c) return;
  if (--c->refs > 0) return;
  // Last reference: release device resources.  (The reference keeps its singleton alive for the process;
  // releasing here keeps create/destroy loops leak-free and a later create simply rebuilds it.)
  g_ctxs[c->device] = nullptr;
  DeviceGuard dg(c->device);
  cudaStreamSynchronize(c->stream);
  for (auto& s : c->scratch) s.release();
  cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1);
  for (auto* v : {&c->ev_in, &c->ev_k0, &c->ev_k1}) { for (cudaEvent_t ev : *v) cudaEventDestroy(ev); v->clear(); }
  if (c->h2d) cudaStreamDestroy(c->h2d);
  if (c->d2h) cudaStreamDestroy(c->d2h);
  cudaStreamDestroy(c->stream);
  cudaGetLastError();
  delete c;
}

mfa_error_t mfa_create_buffer(mfa_context_t context, size_t size_bytes, mfa_buffer_t* buffer) {
  if (!context || !buffer) return MFA_ERROR_INVALID_ARGS;
  *buffer = nullptr;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  Context* ctx = C_(context);
  DeviceGuard dg(ctx->device);
  Buffer* b = new (std::nothrow) Buffer();
  if (!b) return MFA_ERROR_MEMORY_ALLOCATION;
  b->owner = ctx;
  b->bytes = size_bytes;
  size_t alloc = size_bytes ? size_bytes : 1;
  if (cudaHostAlloc(&b->host, alloc, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); delete b; return MFA_ERROR_MEMORY_ALLOCATION; }
  if (cudaMalloc(&b->dev, alloc) != cudaSuccess) { cudaGetLastError(); cudaFreeHost(b->host); delete b; return MFA_ERROR_MEMORY_ALLOCATION; }
  memset(b->host, 0, alloc);
  cudaMemset(b->dev, 0, alloc);
  b->owns_host = b->owns_dev = true;
  b->mirrored = true;
  *buffer = b;
  return MFA_SUCCESS;
}

mfa_error_t mfa_buffer_from_ptr(mfa_context_t context, void* data_ptr, size_t size_bytes, mfa_buffer_t* buffer) {
  if (buffer) *buffer = nullptr;
  return make_buffer(C_(context), data_ptr, size_bytes, false, nullptr, nullptr, 0, buffer);
}

mfa_error_t mfa_buffer_from_ptr_with_strides(mfa_context_t context, void* data_ptr, size_t size_bytes,
                                             const int64_t* shape, const int64_t* strides, uint32_t ndim,
                                             mfa_buffer_t* buffer) {
  if (buffer) *buffer = nullptr;
  return make_buffer(C_(context), data_ptr, size_bytes, false, shape, strides, ndim, buffer);
}

mfa_error_t mfa_buffer_from_mtl_buffer(mfa_context_t context, void* metal_buffer, size_t size_bytes,
                                       mfa_buffer_t* buffer) {
  if (buffer) *buffer = nullptr;
  return make_buffer(C_(context), metal_buffer, size_bytes, true, nullptr, nullptr, 0, buffer);
}

mfa_error_t mfa_buffer_from_mtl_buffer_with_strides(mfa_context_t context, void* metal_buffer, size_t size_bytes,
                                                    const int64_t* shape, const int64_t* strides, uint32_t ndim,
                                                    mfa_buffer_t* buffer) {
  if (buffer) *buffer = nullptr;
  return make_buffer(C_(context), metal_buffer, size_bytes, true, shape, strides, ndim, buffer);
}

void* mfa_buffer_contents(mfa_buffer_t buffer) {
  if (!buffer) return nullptr;
  Buffer* b = B_(buffer);
  return b->host ? b->host : b->dev;
}

void mfa_destroy_buffer(mfa_buffer_t buffer) {
  if (!buffer) return;
  Buffer* b = B_(buffer);
  if (b->registered) cudaHostUnregister(b->host);
  if (b->owns_dev && b->dev) cudaFree(b->dev);
  if (b->owns_host && b->host) cudaFreeHost(b->host);
  cudaGetLastError();
  delete b;
}

mfa_error_t mfa_attention_forward(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal,
    mfa_precision_t input_precision, mfa_precision_t, mfa_precision_t output_precision,
    bool transpose_q, bool transpose_k, bool transpose_v, bool transpose_o,
    const void* mask_ptr, size_t mask_size_bytes, const int64_t* mask_shape, const int64_t* mask_strides,
    uint32_t mask_ndim, mfa_mask_type_t mask_type, mfa_mask_scalar_t mask_scalar_type) {
  if (!context || !q || !k || !v || !out) return MFA_ERROR_INVALID_ARGS;
  FwdArgs a{B_(q), B_(k), B_(v), B_(out), nullptr, batch_size, seq_len_q, seq_len_kv, num_heads, head_dim,
            softmax_scale, causal, -1, header_precision_to_dtype(input_precision),
            header_precision_to_dtype(output_precision), transpose_q, transpose_k, transpose_v, transpose_o,
            MaskArgs{mask_ptr, mask_size_bytes, mask_shape, mask_strides, mask_ndim, mask_type, mask_scalar_type},
            nullptr, false};
  return forward_core(C_(context), a);
}

mfa_error_t mfa_attention_forward_str(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal,
    const char* input_precision, const char*, const char* output_precision,
    bool transpose_q, bool transpose_k, bool transpose_v, bool transpose_o,
    const void* mask_ptr, size_t mask_size_bytes, const int64_t* mask_shape, const int64_t* mask_strides,
    uint32_t mask_ndim, mfa_mask_type_t mask_type, mfa_mask_scalar_t mask_scalar_type) {
  if (!context || !q || !k || !v || !out) return MFA_ERROR_INVALID_ARGS;
  FwdArgs a{B_(q), B_(k), B_(v), B_(out), nullptr, batch_size, seq_len_q, seq_len_kv, num_heads, head_dim,
            softmax_scale, causal, -1, parse_precision_str(input_precision), parse_precision_str(output_precision),
            transpose_q, transpose_k, transpose_v, transpose_o,
            MaskArgs{mask_ptr, mask_size_bytes, mask_shape, mask_strides, mask_ndim, mask_type, mask_scalar_type},
            nullptr, false};
  return forward_core(C_(context), a);
}

int32_t mfa_attention_forward_with_lse(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t lse,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t input_precision, int32_t,
    bool transpose_q, bool transpose_k, bool transpose_v, bool transpose_o) {
  if (!context || !q || !k || !v || !out || !lse) return MFA_ERROR_INVALID_ARGS;
  FwdArgs a{B_(q), B_(k), B_(v), B_(out), B_(lse), batch_size, seq_len_q, seq_len_kv, num_heads, head_dim,
            softmax_scale, causal, -1, header_precision_to_dtype(input_precision), kF32,
            transpose_q, transpose_k, transpose_v, transpose_o, MaskArgs{nullptr, 0, nullptr, nullptr, 0, 0, 0},
            nullptr, false};
  return forward_core(C_(context), a);
}

mfa_error_t mfa_attention_forward_ex(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t lse,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t window_size,
    mfa_precision_t input_precision, mfa_precision_t output_precision,
    const void* mask_ptr, size_t mask_size_bytes, const int64_t* mask_shape, const int64_t* mask_strides,
    uint32_t mask_ndim, mfa_mask_type_t mask_type, mfa_mask_scalar_t mask_scalar_type, void* stream) {
  if (!context || !q || !k || !v || !out) return MFA_ERROR_INVALID_ARGS;
  FwdArgs a{B_(q), B_(k), B_(v), B_(out), B_(lse), batch_size, seq_len_q, seq_len_kv, num_heads, head_dim,
            softmax_scale, causal, window_size < 0 ? -1 : window_size, header_precision_to_dtype(input_precision),
            header_precision_to_dtype(output_precision), false, false, false, false,
            MaskArgs{mask_ptr, mask_size_bytes, mask_shape, mask_strides, mask_ndim, mask_type, mask_scalar_type},
            reinterpret_cast<cudaStream_t>(stream), stream != nullptr};
  return forward_core(C_(context), a);
}

// Ring attention step: attention of `seq_len_q` query rows against one visiting K/V block, merged in place into rows
// [acc_row_offset, acc_row_offset + seq_len_q) of every (b, h) of the running fp32 result out_acc [B, H, acc_rows, D] /
// lse_acc [B, H, acc_rows] (log2-domain merge, SURVEY 8e).  Tensor-core operands only (bf16 / fp16, head_dim 64 / 128):
// the merge happens in the kernel epilogue, so no partial O is ever written to HBM.
mfa_error_t mfa_attention_forward_accumulate(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out_acc, mfa_buffer_t lse_acc,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t window_size, mfa_precision_t input_precision,
    uint32_t acc_row_offset, uint32_t acc_rows, void* stream) {
  if (!context || !q || !k || !v || !out_acc || !lse_acc) return MFA_ERROR_INVALID_ARGS;
  Context* ctx = C_(context);
  Buffer *bq = B_(q), *bk = B_(k), *bv = B_(v), *bo = B_(out_acc), *bl = B_(lse_acc);
  const int in_dtype = header_precision_to_dtype(input_precision);
  if (in_dtype != kBF16 && in_dtype != kF16) return MFA_ERROR_INVALID_ARGS;
  if ((uint64_t)acc_row_offset + seq_len_q > acc_rows) return MFA_ERROR_INVALID_ARGS;
  if (bq->mirrored || bk->mirrored || bv->mirrored || bo->mirrored || bl->mirrored) return MFA_ERROR_INVALID_ARGS;
  if (!view_fits(bq, batch_size, num_heads, seq_len_q, head_dim, 2) || !view_fits(bk, batch_size, num_heads, seq_len_kv, head_dim, 2) ||
      !view_fits(bv, batch_size, num_heads, seq_len_kv, head_dim, 2))
    return MFA_ERROR_INVALID_ARGS;
  if (bo->bytes < elems(batch_size, num_heads, acc_rows, head_dim) * 4 || bl->bytes < (size_t)batch_size * num_heads * acc_rows * 4)
    return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  if (batch_size == 0 || num_heads == 0 || seq_len_q == 0 || seq_len_kv == 0) return MFA_SUCCESS;
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  cudaStream_t st = stream ? reinterpret_cast<cudaStream_t>(stream) : ctx->stream;
  AttnParams p;
  init_params(p, batch_size, num_heads, seq_len_q, seq_len_kv, head_dim, softmax_scale, causal, window_size < 0 ? -1 : window_size);
  p.q = view_of(bq, num_heads, seq_len_q, head_dim, false);
  p.k = view_of(bk, num_heads, seq_len_kv, head_dim, false);
  p.v = view_of(bv, num_heads, seq_len_kv, head_dim, false);
  const int64_t D = head_dim, T = acc_rows;
  p.o = TensorView{reinterpret_cast<float*>(bo->dev) + (size_t)acc_row_offset * D, (int64_t)num_heads * T * D, T * D, D, 1};
  p.lse = reinterpret_cast<float*>(bl->dev) + acc_row_offset;
  p.lse_sh = T;
  p.accumulate = 1;
  p.in_dtype = in_dtype; p.o_dtype = kF32;
  if (!fwd_tc_eligible(p)) return MFA_ERROR_INVALID_ARGS;
  Timer tm(ctx, st, stream == nullptr);
  cudaError_t e = launch_fwd_tc(p, st);
  tm.stop();
  ctx->last_kernel = g_last_kernel;
  if (e != cudaSuccess) return cuda_fail(e, "forward accumulate launch");
  if (!stream) {
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return cuda_fail(e, "forward accumulate sync");
    tm.read();
  }
  return MFA_SUCCESS;
}

mfa_error_t mfa_attention_encode_mtl(
    mfa_context_t context, void* command_buffer,
    void* q_buffer, int64_t q_offset, const int64_t* q_strides,
    void* k_buffer, int64_t k_offset, const int64_t* k_strides,
    void* v_buffer, int64_t v_offset, const int64_t* v_strides,
    void* out_buffer, int64_t out_offset,
    void* mask_buffer, int64_t mask_offset, const int64_t* mask_shape, const int64_t* mask_strides,
    uint32_t mask_ndim, mfa_mask_type_t mask_type, mfa_mask_scalar_t mask_scalar_type,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, const char* input_precision, const char*) {
  if (!context || !q_buffer || !k_buffer || !v_buffer || !out_buffer) return MFA_ERROR_INVALID_ARGS;
  const int dt = parse_precision_str(input_precision);
  if (!valid_float_dtype(dt)) return MFA_ERROR_INVALID_ARGS;
  // Raw device pointers + byte offsets: wrap them in transient views (no ownership, no mirrors).
  Buffer qb, kb, vb, ob;
  auto wrap = [&](Buffer& b, void* base, int64_t off, const int64_t* strides, uint32_t S, size_t esz) {
    b.dev = reinterpret_cast<char*>(base) + off;
    b.bytes = elems(batch_size, num_heads, S, head_dim) * esz;
    if (strides) {
      b.ndim = 4;
      b.shape[0] = batch_size; b.shape[1] = num_heads; b.shape[2] = S; b.shape[3] = head_dim;
      for (int i = 0; i < 4; ++i) b.strides[i] = strides[i];
    }
  };
  wrap(qb, q_buffer, q_offset, q_strides, seq_len_q, dtype_bytes(dt));
  wrap(kb, k_buffer, k_offset, k_strides, seq_len_kv, dtype_bytes(dt));
  wrap(vb, v_buffer, v_offset, v_strides, seq_len_kv, dtype_bytes(dt));
  wrap(ob, out_buffer, out_offset, nullptr, seq_len_q, 4);
  size_t mask_bytes = 0;
  const void* mptr = nullptr;
  if (mask_buffer && mask_type != MFA_MASK_TYPE_NONE && mask_ndim && mask_shape) {
    mptr = reinterpret_cast<char*>(mask_buffer) + mask_offset;
    size_t esz = mask_type == MFA_MASK_TYPE_BOOL ? 1 : (mask_scalar_type == MFA_MASK_SCALAR_FP32 ? 4 : 2);
    int64_t span = 1;
    for (uint32_t i = 0; i < mask_ndim; ++i)
      span += (mask_shape[i] - 1) * (mask_strides ? mask_strides[i] : 0);
    if (!mask_strides) { span = 1; for (uint32_t i = 0; i < mask_ndim; ++i) span *= mask_shape[i]; }
    mask_bytes = (size_t)span * esz;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(command_buffer);
  FwdArgs a{&qb, &kb, &vb, &ob, nullptr, batch_size, seq_len_q, seq_len_kv, num_heads, head_dim, softmax_scale, causal,
            -1, dt, kF32, false, false, false, false,
            MaskArgs{mptr, mask_bytes, mask_shape, mask_strides, mask_ndim, mask_type, mask_scalar_type}, st, true};
  return forward_core(C_(context), a);
}

mfa_error_t mfa_attention_backward(
    mfa_context_t context,
    mfa_buffer_t dout, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t softmax_lse,
    mfa_buffer_t dq, mfa_buffer_t dk, mfa_buffer_t dv, mfa_buffer_t d_buffer,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, mfa_precision_t input_precision, mfa_precision_t,
    bool transpose_q, bool transpose_k, bool transpose_v, bool transpose_o) {
  if (!context || !dout || !q || !k || !v || !out || !softmax_lse || !dq || !dk || !dv) return MFA_ERROR_INVALID_ARGS;
  const int dt = header_precision_to_dtype(input_precision);
  if (!valid_float_dtype(dt)) return MFA_ERROR_INVALID_ARGS;
  QuantView none{nullptr, 1.f, 0, 0};
  BwdArgs a{B_(dout), B_(q), B_(k), B_(v), B_(out), B_(softmax_lse), B_(dq), B_(dk), B_(dv), B_(d_buffer),
            batch_size, seq_len_q, seq_len_kv, num_heads, num_heads, head_dim, softmax_scale, causal, -1,
            dt, dt, transpose_q, transpose_k, transpose_v, transpose_o,
            MaskArgs{nullptr, 0, nullptr, nullptr, 0, 0, 0}, none, none, none, nullptr, false, true, true};
  // dO arrives in the input precision (MetalFlashAttentionFn::backward passes grad in q's dtype).
  return backward_core(C_(context), a);
}

mfa_error_t mfa_attention_backward_ex(
    mfa_context_t context,
    mfa_buffer_t dout, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t softmax_lse,
    mfa_buffer_t dq, mfa_buffer_t dk, mfa_buffer_t dv, mfa_buffer_t d_buffer,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t window_size, mfa_precision_t input_precision,
    const void* mask_ptr, size_t mask_size_bytes, const int64_t* mask_shape, const int64_t* mask_strides,
    uint32_t mask_ndim, mfa_mask_type_t mask_type, mfa_mask_scalar_t mask_scalar_type, void* stream) {
  if (!context || !dout || !q || !k || !v || !out || !softmax_lse || !dq || !dk || !dv) return MFA_ERROR_INVALID_ARGS;
  const int dt = header_precision_to_dtype(input_precision);
  if (!valid_float_dtype(dt)) return MFA_ERROR_INVALID_ARGS;
  QuantView none{nullptr, 1.f, 0, 0};
  BwdArgs a{B_(dout), B_(q), B_(k), B_(v), B_(out), B_(softmax_lse), B_(dq), B_(dk), B_(dv), B_(d_buffer),
            batch_size, seq_len_q, seq_len_kv, num_heads, num_heads, head_dim, softmax_scale, causal,
            window_size < 0 ? -1 : window_size, dt, dt, false, false, false, false,
            MaskArgs{mask_ptr, mask_size_bytes, mask_shape, mask_strides, mask_ndim, mask_type, mask_scalar_type},
            none, none, none, reinterpret_cast<cudaStream_t>(stream), stream != nullptr, true, true};
  return backward_core(C_(context), a);
}

mfa_error_t mfa_attention_forward_varlen(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t lse,
    mfa_buffer_t cu_seqlens_q, mfa_buffer_t cu_seqlens_k, uint32_t num_seqs, uint32_t total_q, uint32_t total_k,
    uint32_t num_heads, uint32_t num_kv_heads, uint16_t head_dim, float softmax_scale, bool causal, int32_t window_size,
    mfa_precision_t input_precision, mfa_precision_t output_precision, void* stream) {
  if (!context || !q || !k || !v || !out) return MFA_ERROR_INVALID_ARGS;
  if (mfa_error_t e = check_segments(B_(cu_seqlens_q), B_(cu_seqlens_k), num_seqs, total_q, total_k); e != MFA_SUCCESS) return e;
  FwdArgs a{B_(q), B_(k), B_(v), B_(out), B_(lse), 1, total_q, total_k, num_heads, head_dim,
            softmax_scale, causal, window_size < 0 ? -1 : window_size, header_precision_to_dtype(input_precision),
            header_precision_to_dtype(output_precision), false, false, false, false,
            MaskArgs{nullptr, 0, nullptr, nullptr, 0, 0, 0}, reinterpret_cast<cudaStream_t>(stream), stream != nullptr,
            num_kv_heads, B_(cu_seqlens_q), B_(cu_seqlens_k), num_seqs};
  return forward_core(C_(context), a);
}

mfa_error_t mfa_attention_backward_varlen(
    mfa_context_t context, mfa_buffer_t dout, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    mfa_buffer_t softmax_lse, mfa_buffer_t dq, mfa_buffer_t dk, mfa_buffer_t dv, mfa_buffer_t d_buffer,
    mfa_buffer_t cu_seqlens_q, mfa_buffer_t cu_seqlens_k, uint32_t num_seqs, uint32_t total_q, uint32_t total_k,
    uint32_t num_heads, uint32_t num_kv_heads, uint16_t head_dim, float softmax_scale, bool causal, int32_t window_size,
    mfa_precision_t input_precision, void* stream) {
  if (!context || !dout || !q || !k || !v || !out || !softmax_lse || !dq || !dk || !dv) return MFA_ERROR_INVALID_ARGS;
  if (mfa_error_t e = check_segments(B_(cu_seqlens_q), B_(cu_seqlens_k), num_seqs, total_q, total_k); e != MFA_SUCCESS) return e;
  const int dt = header_precision_to_dtype(input_precision);
  if (!valid_float_dtype(dt)) return MFA_ERROR_INVALID_ARGS;
  QuantView none{nullptr, 1.f, 0, 0};
  BwdArgs a{B_(dout), B_(q), B_(k), B_(v), B_(out), B_(softmax_lse), B_(dq), B_(dk), B_(dv), B_(d_buffer),
            1, total_q, total_k, num_heads, num_kv_heads ? num_kv_heads : num_heads, head_dim, softmax_scale, causal,
            window_size < 0 ? -1 : window_size, dt, dt, false, false, false, false,
            MaskArgs{nullptr, 0, nullptr, nullptr, 0, 0, 0}, none, none, none, reinterpret_cast<cudaStream_t>(stream),
            stream != nullptr, true, true, B_(cu_seqlens_q), B_(cu_seqlens_k), num_seqs};
  return backward_core(C_(context), a);
}

// The cache geometry shared by the K/V-cache attention calls and mfa_kvcache_append.  Sq is seq_len_q, or with packed
// (cu_seqlens_q) rows the largest number of new tokens of a sequence, total_q the number of packed rows.
struct KvCacheShape {
  uint32_t B, Sq, total_q, H, Hkv, D, cap, page_size, num_pages;
  int dtype;
  bool packed, paged;
};

// Scalar arguments, checked before anything is known about the device.
static bool kvcache_shape_ok(const KvCacheShape& s, mfa_buffer_t block_table) {
  if (s.dtype != kBF16 && s.dtype != kF16) return false;
  if (s.B == 0 || s.Sq == 0 || s.H == 0 || s.H % s.Hkv || s.H / s.Hkv > 128 || s.D < 8 || s.D > 128 || (s.D & 7) || s.cap == 0) return false;
  if (s.B > 65535 || s.Sq > 0x7fffffffu || s.H > 65535 || s.cap > 0x7fffff80u) return false;
  if (s.packed && (s.total_q == 0 || s.total_q > 0x7fffffffu || s.Sq > s.total_q)) return false;
  if (s.paged ? (!block_table || (s.page_size & 15) || s.cap % s.page_size || s.num_pages == 0 || s.num_pages > 0x7fffffffu)
              : block_table != nullptr)
    return false;
  return true;
}

// The caches, cache_seqlens, block_table and cu_seqlens_q handles cover their shapes; offsets, lengths (at most max_len) and page
// ids the host can read are checked here.  Device-resident ones are left to the kernels, which clamp them.
static mfa_error_t check_kvcache_arrays(const KvCacheShape& s, const Buffer* bk, const Buffer* bv, const Buffer* bs, const Buffer* bt,
                                        const Buffer* bc, uint32_t max_len) {
  const uint32_t B = s.B, cap = s.cap;
  if (s.paged) {
    const size_t pool = (size_t)s.num_pages * s.page_size * s.Hkv * s.D * 2;
    if (bk->ndim || bv->ndim || bk->bytes < pool || bv->bytes < pool) return MFA_ERROR_INVALID_ARGS;
    if (bt->ndim || bt->bytes < (size_t)B * (cap / s.page_size) * 4) return MFA_ERROR_INVALID_ARGS;
  } else if (!view_fits(bk, B, s.Hkv, cap, s.D, 2) || !view_fits(bv, B, s.Hkv, cap, s.D, 2)) {
    return MFA_ERROR_INVALID_ARGS;
  }
  if (bs->ndim || bs->bytes < (size_t)B * 4) return MFA_ERROR_INVALID_ARGS;
  if (s.packed && (bc->ndim || bc->bytes < ((size_t)B + 1) * 4)) return MFA_ERROR_INVALID_ARGS;
  if (s.packed && bc->host) {
    const int32_t* cu = reinterpret_cast<const int32_t*>(bc->host);
    if (cu[0] != 0 || cu[B] != (int64_t)s.total_q) return MFA_ERROR_INVALID_ARGS;
    for (uint32_t b = 0; b < B; ++b)
      if (cu[b + 1] < cu[b] || (int64_t)cu[b + 1] - cu[b] > (int64_t)s.Sq) return MFA_ERROR_INVALID_ARGS;
  }
  if (bs->host) {
    const int32_t* len = reinterpret_cast<const int32_t*>(bs->host);
    for (uint32_t b = 0; b < B; ++b)
      if (len[b] < 0 || (uint32_t)len[b] > max_len) return MFA_ERROR_INVALID_ARGS;
  }
  if (s.paged && bt->host) {
    const int32_t* ids = reinterpret_cast<const int32_t*>(bt->host);
    for (size_t i = 0, n = (size_t)B * (cap / s.page_size); i < n; ++i)
      if (ids[i] < 0 || (uint32_t)ids[i] >= s.num_pages) return MFA_ERROR_INVALID_ARGS;
  }
  return MFA_SUCCESS;
}

// mfa_attention_forward_kvcache (cu_seqlens_q null: seq_len_q new tokens per sequence) and
// mfa_attention_forward_kvcache_varlen (sequence b owns query rows [cu[b], cu[b+1]) of total_q, at most seq_len_q of them).
static mfa_error_t kvcache_forward(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k_cache, mfa_buffer_t v_cache, mfa_buffer_t out, mfa_buffer_t lse,
    mfa_buffer_t cu_seqlens_q, mfa_buffer_t cache_seqlens, mfa_buffer_t block_table,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t total_q, uint32_t num_heads, uint32_t num_kv_heads, uint16_t head_dim,
    uint32_t cache_capacity, uint32_t page_size, uint32_t num_pages,
    float softmax_scale, bool causal, int32_t window_size,
    mfa_precision_t input_precision, mfa_precision_t output_precision, void* stream) {
  const uint32_t B = batch_size, Sq = seq_len_q, H = num_heads, Hkv = num_kv_heads ? num_kv_heads : num_heads, D = head_dim;
  const uint32_t cap = cache_capacity;
  const bool packed = cu_seqlens_q != nullptr;
  const int dt = header_precision_to_dtype(input_precision), odt = header_precision_to_dtype(output_precision);
  if (!valid_float_dtype(odt) || !(softmax_scale > 0.f)) return MFA_ERROR_INVALID_ARGS;
  const KvCacheShape shape{B, Sq, total_q, H, Hkv, D, cap, page_size, num_pages, dt, packed, page_size > 0};
  if (!kvcache_shape_ok(shape, block_table)) return MFA_ERROR_INVALID_ARGS;
  const bool paged = shape.paged;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  Buffer *bq = B_(q), *bk = B_(k_cache), *bv = B_(v_cache), *bo = B_(out), *bl = B_(lse), *bs = B_(cache_seqlens), *bt = B_(block_table);
  Buffer* bc = B_(cu_seqlens_q);
  // Q / O / L: [B, H, Sq] rows, or the [1, H, total_q] packed rows
  const uint32_t qB = packed ? 1 : B, qS = packed ? total_q : Sq;
  if (!view_fits(bq, qB, H, qS, D, 2) || !view_fits(bo, qB, H, qS, D, dtype_bytes(odt))) return MFA_ERROR_INVALID_ARGS;
  if (bl && bl->bytes < (size_t)qB * H * qS * 4) return MFA_ERROR_INVALID_ARGS;
  if (mfa_error_t e = check_kvcache_arrays(shape, bk, bv, bs, bt, bc, cap)) return e;
  const bool async = stream != nullptr;
  if (async && (bq->mirrored || bk->mirrored || bv->mirrored || bo->mirrored || (bl && bl->mirrored) || bs->mirrored || (bt && bt->mirrored) ||
                (bc && bc->mirrored)))
    return MFA_ERROR_INVALID_ARGS;

  Context* ctx = C_(context);
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  KvCacheParams p;
  p.q = view_of(bq, H, qS, D, false);
  p.o = view_of(bo, H, qS, D, false);
  p.k = view_of(bk, Hkv, cap, D, false);
  p.v = view_of(bv, Hkv, cap, D, false);
  p.lse = bl ? reinterpret_cast<float*>(bl->dev) : nullptr;
  p.seqlens = reinterpret_cast<const int*>(bs->dev);
  p.block_table = paged ? reinterpret_cast<const int*>(bt->dev) : nullptr;
  p.cu_q = packed ? reinterpret_cast<const int*>(bc->dev) : nullptr;
  p.B = (int)B; p.H = (int)H; p.Hkv = (int)Hkv; p.Sq = (int)Sq; p.D = (int)D; p.cap = (int)cap;
  p.page_size = (int)page_size; p.num_pages = (int)num_pages;
  p.total_q = packed ? (int)total_q : 0;
  p.scale = softmax_scale; p.causal = causal ? 1 : 0; p.window = window_size < 0 ? -1 : window_size;
  p.in_dtype = dt; p.o_dtype = odt;
  // TMA: 16-byte aligned bases and outer strides; out only needs unit stride along D (the combine kernel stores elements)
  if (!tc::view_ok(p.q, H, qB) || p.o.sd != 1 || (!paged && (!tc::view_ok(p.k, Hkv, B) || !tc::view_ok(p.v, Hkv, B))) ||
      (paged && ((reinterpret_cast<uintptr_t>(bk->dev) | reinterpret_cast<uintptr_t>(bv->dev)) & 15)))
    return MFA_ERROR_INVALID_ARGS;
  static int sm_count[kMaxDevices] = {0};
  if (!sm_count[ctx->device] && cudaDeviceGetAttribute(&sm_count[ctx->device], cudaDevAttrMultiProcessorCount, ctx->device) != cudaSuccess) {
    cudaGetLastError();
    sm_count[ctx->device] = 148;
  }
  const KvCachePlan plan = kvcache_plan(p, sm_count[ctx->device]);
  const size_t bytes = plan.o_bytes + plan.l_bytes;

  cudaStream_t st = async ? reinterpret_cast<cudaStream_t>(stream) : ctx->stream;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (async && cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); return MFA_ERROR_EXECUTION_FAILED; }
  ScratchScope scope(ctx, st);
  void* scratch = nullptr;
  Scratch& ksc = ctx->scratch[Context::kKvSplit];
  if (cs != cudaStreamCaptureStatusNone) {
    // inside a graph capture: no allocation.  The graph keeps the block (Scratch::captured) and orders itself against other
    // users of it through external event nodes: a replay waits for the last use recorded before its launch and records its own.
    if (ksc.cap < bytes) return MFA_ERROR_MEMORY_ALLOCATION;
    if (!ksc.ev && cudaEventCreateWithFlags(&ksc.ev, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return MFA_ERROR_EXECUTION_FAILED; }
    if (ksc.used && cudaStreamWaitEvent(st, ksc.ev, cudaEventWaitExternal) != cudaSuccess) { cudaGetLastError(); return MFA_ERROR_EXECUTION_FAILED; }
    scratch = ksc.ptr;
  } else if (!(scratch = scope.take(Context::kKvSplit, bytes))) {
    return MFA_ERROR_MEMORY_ALLOCATION;
  }
  Sync sync{ctx, st, async, {}};
  cudaError_t e;
  if ((e = sync.in(bq)) != cudaSuccess || (e = sync.in(bk)) != cudaSuccess || (e = sync.in(bv)) != cudaSuccess ||
      (e = sync.in(bs)) != cudaSuccess || (e = sync.in(bt)) != cudaSuccess || (e = sync.in(bc)) != cudaSuccess)
    return cuda_fail(e, "h2d");
  Timer tm(ctx, st, !async);
  e = launch_fwd_kvcache(p, plan, scratch, st);
  if (e == cudaSuccess && cs != cudaStreamCaptureStatusNone) {
    e = cudaEventRecordWithFlags(ksc.ev, st, cudaEventRecordExternal);
    ksc.captured = true; ksc.used = true;
    ksc.last = nullptr;                // every later call, on any stream, waits for the replays' record
  }
  tm.stop();
  ctx->last_kernel = g_last_kernel;
  if (e != cudaSuccess) return cuda_fail(e, "kvcache forward launch");
  sync.out(bo); sync.out(bl);
  if ((e = sync.finish()) != cudaSuccess) return cuda_fail(e, "kvcache forward sync");
  tm.read();
  return MFA_SUCCESS;
}

mfa_error_t mfa_attention_forward_kvcache(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k_cache, mfa_buffer_t v_cache, mfa_buffer_t out, mfa_buffer_t lse,
    mfa_buffer_t cache_seqlens, mfa_buffer_t block_table,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t num_heads, uint32_t num_kv_heads, uint16_t head_dim,
    uint32_t cache_capacity, uint32_t page_size, uint32_t num_pages,
    float softmax_scale, bool causal, int32_t window_size,
    mfa_precision_t input_precision, mfa_precision_t output_precision, void* stream) {
  if (!context || !q || !k_cache || !v_cache || !out || !cache_seqlens) return MFA_ERROR_INVALID_ARGS;
  return kvcache_forward(context, q, k_cache, v_cache, out, lse, nullptr, cache_seqlens, block_table, batch_size, seq_len_q, 0,
                         num_heads, num_kv_heads, head_dim, cache_capacity, page_size, num_pages, softmax_scale, causal, window_size,
                         input_precision, output_precision, stream);
}

mfa_error_t mfa_attention_forward_kvcache_varlen(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k_cache, mfa_buffer_t v_cache, mfa_buffer_t out, mfa_buffer_t lse,
    mfa_buffer_t cu_seqlens_q, mfa_buffer_t cache_seqlens, mfa_buffer_t block_table,
    uint32_t num_seqs, uint32_t total_q, uint32_t max_seqlen_q, uint32_t num_heads, uint32_t num_kv_heads, uint16_t head_dim,
    uint32_t cache_capacity, uint32_t page_size, uint32_t num_pages,
    float softmax_scale, bool causal, int32_t window_size,
    mfa_precision_t input_precision, mfa_precision_t output_precision, void* stream) {
  if (!context || !q || !k_cache || !v_cache || !out || !cu_seqlens_q || !cache_seqlens) return MFA_ERROR_INVALID_ARGS;
  return kvcache_forward(context, q, k_cache, v_cache, out, lse, cu_seqlens_q, cache_seqlens, block_table, num_seqs, max_seqlen_q,
                         total_q, num_heads, num_kv_heads, head_dim, cache_capacity, page_size, num_pages, softmax_scale, causal,
                         window_size, input_precision, output_precision, stream);
}

mfa_error_t mfa_kvcache_append(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t q_out, mfa_buffer_t k_new, mfa_buffer_t v_new,
    mfa_buffer_t k_cache, mfa_buffer_t v_cache,
    mfa_buffer_t cu_seqlens_q, mfa_buffer_t cache_seqlens, mfa_buffer_t block_table,
    mfa_buffer_t rotary_cos, mfa_buffer_t rotary_sin, uint32_t rotary_rows, uint16_t rotary_dim, bool rotary_interleaved,
    uint32_t num_seqs, uint32_t total_q, uint32_t max_seqlen_q, uint32_t num_heads, uint32_t num_kv_heads, uint16_t head_dim,
    uint32_t cache_capacity, uint32_t page_size, uint32_t num_pages,
    mfa_precision_t input_precision, void* stream) {
  if (!context || !k_new || !v_new || !k_cache || !v_cache || !cache_seqlens) return MFA_ERROR_INVALID_ARGS;
  const bool packed = cu_seqlens_q != nullptr, rotary = rotary_cos != nullptr;
  const uint32_t B = num_seqs, Sq = max_seqlen_q, H = num_heads, Hkv = num_kv_heads ? num_kv_heads : num_heads, D = head_dim;
  if ((q == nullptr) != (q_out == nullptr) || (q && !rotary) || (rotary_sin != nullptr) != rotary) return MFA_ERROR_INVALID_ARGS;
  if (rotary ? (rotary_dim == 0 || (rotary_dim & 15) || rotary_dim > D || rotary_rows == 0 || rotary_rows > 0x7fffffffu)
             : rotary_dim != 0)
    return MFA_ERROR_INVALID_ARGS;
  const KvCacheShape shape{B, Sq, total_q, H, Hkv, D, cache_capacity, page_size, num_pages,
                           header_precision_to_dtype(input_precision), packed, page_size > 0};
  if (!kvcache_shape_ok(shape, block_table)) return MFA_ERROR_INVALID_ARGS;
  const uint64_t tokens = packed ? total_q : (uint64_t)B * Sq;        // one CTA per token
  if (tokens > 0x7fffffffu) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  Buffer *bq = B_(q), *bqo = B_(q_out), *bkn = B_(k_new), *bvn = B_(v_new), *bk = B_(k_cache), *bv = B_(v_cache);
  Buffer *bc = B_(cu_seqlens_q), *bs = B_(cache_seqlens), *bt = B_(block_table), *bcos = B_(rotary_cos), *bsin = B_(rotary_sin);
  const uint32_t qB = packed ? 1 : B, qS = packed ? total_q : Sq;
  if (q && (!view_fits(bq, qB, H, qS, D, 2) || !view_fits(bqo, qB, H, qS, D, 2))) return MFA_ERROR_INVALID_ARGS;
  if (!view_fits(bkn, qB, Hkv, qS, D, 2) || !view_fits(bvn, qB, Hkv, qS, D, 2)) return MFA_ERROR_INVALID_ARGS;
  const size_t table_bytes = (size_t)rotary_rows * (rotary_dim / 2) * 4;
  if (rotary && (bcos->ndim || bsin->ndim || bcos->bytes < table_bytes || bsin->bytes < table_bytes)) return MFA_ERROR_INVALID_ARGS;
  if (mfa_error_t e = check_kvcache_arrays(shape, bk, bv, bs, bt, bc, rotary ? std::min(cache_capacity, rotary_rows) : cache_capacity))
    return e;
  const bool async = stream != nullptr;
  const Buffer* all[] = {bq, bqo, bkn, bvn, bk, bv, bc, bs, bt, bcos, bsin};
  if (async)
    for (const Buffer* b : all)
      if (b && b->mirrored) return MFA_ERROR_INVALID_ARGS;

  Context* ctx = C_(context);
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  KvAppendParams p;
  memset(&p, 0, sizeof(p));
  if (q) {
    p.q = view_of(bq, H, qS, D, false);
    p.q_out = view_of(bqo, H, qS, D, false);
  }
  p.k_new = view_of(bkn, Hkv, qS, D, false);
  p.v_new = view_of(bvn, Hkv, qS, D, false);
  p.k = view_of(bk, Hkv, cache_capacity, D, false);
  p.v = view_of(bv, Hkv, cache_capacity, D, false);
  p.seqlens = reinterpret_cast<const int*>(bs->dev);
  p.block_table = shape.paged ? reinterpret_cast<const int*>(bt->dev) : nullptr;
  p.cu_q = packed ? reinterpret_cast<const int*>(bc->dev) : nullptr;
  p.cos_t = rotary ? reinterpret_cast<const float*>(bcos->dev) : nullptr;
  p.sin_t = rotary ? reinterpret_cast<const float*>(bsin->dev) : nullptr;
  p.rotary_rows = (int)rotary_rows; p.rotary_dim = rotary_dim; p.interleaved = rotary_interleaved ? 1 : 0;
  p.B = (int)B; p.H = (int)H; p.Hkv = (int)Hkv; p.Sq = (int)Sq; p.D = (int)D; p.cap = (int)cache_capacity;
  p.page_size = (int)page_size; p.num_pages = (int)num_pages;
  p.total_q = (int)tokens; p.dtype = shape.dtype;
  // 16-byte vector accesses: aligned bases and outer strides, unit stride along D
  if ((q && (!tc::view_ok(p.q, H, qB) || !tc::view_ok(p.q_out, H, qB))) || !tc::view_ok(p.k_new, Hkv, qB) ||
      !tc::view_ok(p.v_new, Hkv, qB) || (!shape.paged && (!tc::view_ok(p.k, Hkv, B) || !tc::view_ok(p.v, Hkv, B))) ||
      ((reinterpret_cast<uintptr_t>(bk->dev) | reinterpret_cast<uintptr_t>(bv->dev)) & 15) ||
      (rotary && ((reinterpret_cast<uintptr_t>(bcos->dev) | reinterpret_cast<uintptr_t>(bsin->dev)) & 15)))
    return MFA_ERROR_INVALID_ARGS;

  cudaStream_t st = async ? reinterpret_cast<cudaStream_t>(stream) : ctx->stream;
  Sync sync{ctx, st, async, {}};
  cudaError_t e = cudaSuccess;
  // the caches and q_out are copied in too: rows the kernel does not write must come back unchanged
  for (const Buffer* b : all)
    if (e == cudaSuccess) e = sync.in(const_cast<Buffer*>(b));
  if (e != cudaSuccess) return cuda_fail(e, "h2d");
  Timer tm(ctx, st, !async);
  e = launch_kvcache_append(p, st);
  tm.stop();
  ctx->last_kernel = g_last_kernel;
  if (e != cudaSuccess) return cuda_fail(e, "kvcache append launch");
  sync.out(bk); sync.out(bv); sync.out(bqo);
  if ((e = sync.finish()) != cudaSuccess) return cuda_fail(e, "kvcache append sync");
  tm.read();
  return MFA_SUCCESS;
}

// ---- quantised forward family ---------------------------------------------------------------------
static mfa_error_t quantized_forward_common(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t B, uint32_t Sq, uint32_t Skv, uint32_t H, uint16_t D, float scale, bool causal,
    float q_scale, int32_t q_zp, float k_scale, int32_t k_zp, float v_scale, int32_t v_zp,
    int q_prec, int k_prec, int v_prec, int out_prec, int granularity, uint32_t qb, uint32_t kb, uint32_t vb) {
  if (!context || !q || !k || !v || !out) return MFA_ERROR_INVALID_ARGS;
  int dq = header_precision_to_dtype(q_prec), dk = header_precision_to_dtype(k_prec), dv = header_precision_to_dtype(v_prec);
  if (dq < 0 || dk < 0 || dv < 0) return MFA_ERROR_INVALID_ARGS;
  // target integer width = the narrowest integer type any operand names (none -> plain floating point attention)
  int target = -1;
  for (int d : {dq, dk, dv}) if (d == kI8 || d == kI4) target = (target == kI4 || d == kI4) ? kI4 : kI8;
  // pre-quantised operands of different widths cannot share one kernel instantiation
  for (int d : {dq, dk, dv}) if ((d == kI8 || d == kI4) && d != target) return MFA_ERROR_INVALID_ARGS;
  auto blk = [&](uint32_t b) -> uint32_t {
    if (granularity == 0) return 0;          // per tensor
    if (granularity == 1) return 1;          // per row
    return b ? b : 64;                       // block / hybrid
  };
  QFwdArgs a{QOperand{B_(q), dq, q_scale, q_zp, blk(qb)}, QOperand{B_(k), dk, k_scale, k_zp, blk(kb)},
             QOperand{B_(v), dv, v_scale, v_zp, blk(vb)}, B_(out), nullptr, nullptr, B, Sq, Skv, H, D, scale, causal,
             target, header_precision_to_dtype(out_prec), granularity == 1};
  if (target < 0) {
    // no integer operand at all: floating-point attention; all three must share a dtype
    if (dq != dk || dk != dv) return MFA_ERROR_INVALID_ARGS;
    FwdArgs f{B_(q), B_(k), B_(v), B_(out), nullptr, B, Sq, Skv, H, D, scale, causal, -1, dq,
              header_precision_to_dtype(out_prec), false, false, false, false,
              MaskArgs{nullptr, 0, nullptr, nullptr, 0, 0, 0}, nullptr, false};
    return forward_core(C_(context), f);
  }
  return qforward_core(C_(context), a);
}

mfa_error_t mfa_attention_forward_quantized(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    mfa_precision_t q_precision, mfa_precision_t k_precision, mfa_precision_t v_precision,
    mfa_precision_t output_precision, bool, bool, bool, bool) {
  return quantized_forward_common(context, q, k, v, out, batch_size, seq_len_q, seq_len_kv, num_heads, head_dim,
                                  softmax_scale, causal, q_scale, q_zero_point, k_scale, k_zero_point, v_scale,
                                  v_zero_point, q_precision, k_precision, v_precision, output_precision, 0, 0, 0, 0);
}

mfa_error_t mfa_attention_forward_quantized_unified(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    mfa_precision_t q_precision, mfa_precision_t k_precision, mfa_precision_t v_precision,
    mfa_precision_t output_precision, int32_t granularity,
    uint32_t q_block_size, uint32_t k_block_size, uint32_t v_block_size, bool, bool, bool, bool, bool, bool) {
  if (granularity < 0 || granularity > 3) return MFA_ERROR_INVALID_ARGS;
  return quantized_forward_common(context, q, k, v, out, batch_size, seq_len_q, seq_len_kv, num_heads, head_dim,
                                  softmax_scale, causal, q_scale, q_zero_point, k_scale, k_zero_point, v_scale,
                                  v_zero_point, q_precision, k_precision, v_precision, output_precision, granularity,
                                  q_block_size, k_block_size, v_block_size);
}

mfa_error_t mfa_attention_forward_quantized_enhanced(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    mfa_precision_t q_precision, mfa_precision_t k_precision, mfa_precision_t v_precision,
    mfa_precision_t output_precision, int32_t granularity,
    uint32_t q_block_size, uint32_t k_block_size, uint32_t v_block_size,
    bool enable_mixed_precision, bool force_symmetric_quantization,
    bool transpose_q, bool transpose_k, bool transpose_v, bool transpose_o) {
  return mfa_attention_forward_quantized_unified(
      context, q, k, v, out, batch_size, seq_len_q, seq_len_kv, num_heads, head_dim, softmax_scale, causal, q_scale,
      q_zero_point, k_scale, k_zero_point, v_scale, v_zero_point, q_precision, k_precision, v_precision,
      output_precision, granularity, q_block_size, k_block_size, v_block_size, enable_mixed_precision,
      force_symmetric_quantization, transpose_q, transpose_k, transpose_v, transpose_o);
}

static mfa_error_t runtime_quantised_forward(mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v,
                                             mfa_buffer_t out, mfa_buffer_t lse, mfa_buffer_t mask, uint32_t B,
                                             uint32_t Sq, uint32_t Skv, uint32_t H, uint16_t D, float scale, bool causal,
                                             int input_prec, int target_prec, int quant_mode, int out_prec) {
  if (!context || !q || !k || !v || !out) return MFA_ERROR_INVALID_ARGS;
  const int in_dt = header_precision_to_dtype(input_prec);
  if (!valid_float_dtype(in_dt)) return MFA_ERROR_INVALID_ARGS;
  if (target_prec != MFA_PRECISION_INT8 && target_prec != MFA_PRECISION_INT4) return MFA_ERROR_INVALID_ARGS;
  if (quant_mode != 0 && quant_mode != 2) return MFA_ERROR_INVALID_ARGS;    // MFABridge+Quantized.swift:268-272
  const uint32_t blk = quant_mode == 2 ? 64 : 0;
  QFwdArgs a{QOperand{B_(q), in_dt, 1.f, 0, blk}, QOperand{B_(k), in_dt, 1.f, 0, blk}, QOperand{B_(v), in_dt, 1.f, 0, blk},
             B_(out), B_(lse), B_(mask), B, Sq, Skv, H, D, scale, causal, target_prec,
             header_precision_to_dtype(out_prec), false};
  return qforward_core(C_(context), a);
}

mfa_error_t mfa_attention_forward_quantized_direct(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, float, int32_t, float, int32_t, float, int32_t,
    int32_t q_precision, int32_t k_precision, int32_t v_precision, int32_t output_precision, bool, bool, bool, bool) {
  return runtime_quantised_forward(context, q, k, v, out, nullptr, nullptr, batch_size, seq_len_q, seq_len_kv, num_heads,
                                   head_dim, softmax_scale, causal, q_precision, k_precision, v_precision,
                                   output_precision);
}

mfa_error_t mfa_multihead_attention_quantized_direct(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, float, int32_t, float, int32_t, float, int32_t,
    int32_t q_precision, int32_t k_precision, int32_t v_precision) {
  return runtime_quantised_forward(context, q, k, v, out, nullptr, nullptr, batch_size, seq_len_q, seq_len_kv, num_heads,
                                   head_dim, softmax_scale, causal, q_precision, k_precision, v_precision,
                                   MFA_PRECISION_FP32);
}

int32_t mfa_quantized_forward_with_lse(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out, mfa_buffer_t lse,
    mfa_buffer_t mask,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t target_precision, int32_t quant_mode, int32_t input_precision) {
  if (!lse) return MFA_ERROR_INVALID_ARGS;
  return runtime_quantised_forward(context, q, k, v, out, lse, mask, batch_size, seq_len_q, seq_len_kv, num_heads,
                                   head_dim, softmax_scale, causal, input_precision, target_precision, quant_mode,
                                   MFA_PRECISION_FP32);
}

// ---- quantised backward family -------------------------------------------------------------------------
static int32_t prequantised_backward(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t output,
    mfa_buffer_t grad_output, mfa_buffer_t logsumexp, mfa_buffer_t grad_query, mfa_buffer_t grad_key,
    mfa_buffer_t grad_value, mfa_buffer_t d_values, uint32_t B, uint32_t Sq, uint32_t Skv, uint32_t H, uint32_t Hkv,
    uint16_t D, float q_scale, int32_t q_zp, float k_scale, int32_t k_zp, float v_scale, int32_t v_zp,
    int32_t q_prec, int32_t k_prec, int32_t v_prec, bool causal, bool want_dq,
    mfa_buffer_t qbs, mfa_buffer_t kbs, mfa_buffer_t vbs, uint32_t qblk, uint32_t kblk, uint32_t vblk) {
  if (!context || !q || !k || !v || !grad_output || !logsumexp || !d_values) return MFA_ERROR_INVALID_ARGS;
  if (want_dq && (!output || !grad_query)) return MFA_ERROR_INVALID_ARGS;
  if (!want_dq && (!grad_key || !grad_value)) return MFA_ERROR_INVALID_ARGS;
  if (q_prec != k_prec || k_prec != v_prec) return MFA_ERROR_INVALID_ARGS;
  const int dt = header_precision_to_dtype(q_prec);
  if (dt < 0) return MFA_ERROR_INVALID_ARGS;
  auto qv = [&](float s, int zp, mfa_buffer_t bs, uint32_t blk) {
    if (bs && blk) return QuantView{reinterpret_cast<const float*>(B_(bs)->dev), 1.f, zp, (int)blk};
    return QuantView{nullptr, s, zp, 0};
  };
  const float scale = 1.0f / sqrtf((float)D);   // these entry points carry no softmax_scale (mfa_ffi.h ref:480-624)
  Context* ctx = C_(context);
  // The dQ entry point also produces D (it owns `output`); the dK/dV entry point consumes d_values as given.
  // backward_core always recomputes D from O and dO, so the kv variant needs O too -- the reference's kv kernel
  // reads D only.  Supply O = nullptr path: recompute is skipped by passing dbuf and want flags.
  Buffer* outb = want_dq ? B_(output) : nullptr;
  if (!want_dq) {
    // dK/dV from the caller's D: run the kv kernel directly.
    if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
    if (D == 0 || D > 256 || H == 0 || Hkv == 0 || H % Hkv) return MFA_ERROR_INVALID_ARGS;
    {
      const size_t nq = elems(B, H, Sq, D), nkv = elems(B, Hkv, Skv, D), rows = (size_t)B * H * Sq;
      if (B_(q)->bytes < packed_bytes(nq, dt) || B_(k)->bytes < packed_bytes(nkv, dt) || B_(v)->bytes < packed_bytes(nkv, dt) ||
          B_(grad_output)->bytes < nq * 4 || B_(logsumexp)->bytes < rows * 4 || B_(d_values)->bytes < rows * 4 ||
          B_(grad_key)->bytes < nkv * 4 || B_(grad_value)->bytes < nkv * 4)
        return MFA_ERROR_INVALID_ARGS;
      auto scales_fit = [&](mfa_buffer_t bs, uint32_t blk, uint32_t Hn, uint32_t S) {
        return !bs || !blk || B_(bs)->bytes >= (size_t)B * Hn * ((S + blk - 1) / blk) * 4;
      };
      if (!scales_fit(qbs, qblk, H, Sq) || !scales_fit(kbs, kblk, Hkv, Skv) || !scales_fit(vbs, vblk, Hkv, Skv))
        return MFA_ERROR_INVALID_ARGS;
    }
    std::lock_guard<std::recursive_mutex> lock(ctx->mu);
    DeviceGuard dg(ctx->device);
    cudaStream_t st = ctx->stream;
    Sync sync{ctx, st, false, {}};
    Buffer* ins[] = {B_(q), B_(k), B_(v), B_(grad_output), B_(logsumexp), B_(d_values), B_(qbs), B_(kbs), B_(vbs)};
    for (Buffer* b : ins) if (b) { cudaError_t e = sync.in(b); if (e != cudaSuccess) return cuda_fail(e, "h2d"); }
    AttnParams p;
    init_params(p, B, H, Sq, Skv, D, scale, causal, -1);
    p.Hkv = (int)Hkv;
    p.q = contiguous_view(B_(q)->dev, H, Sq, D, false);
    p.k = contiguous_view(B_(k)->dev, Hkv, Skv, D, false);
    p.v = contiguous_view(B_(v)->dev, Hkv, Skv, D, false);
    p.d_o = contiguous_view(B_(grad_output)->dev, H, Sq, D, false);
    p.lse = reinterpret_cast<float*>(B_(logsumexp)->dev);
    p.dterm = reinterpret_cast<float*>(B_(d_values)->dev);
    p.in_dtype = dt; p.do_dtype = kF32;
    p.qq = qv(q_scale, q_zp, qbs, qblk); p.qk = qv(k_scale, k_zp, kbs, kblk); p.qv = qv(v_scale, v_zp, vbs, vblk);
    p.dk = reinterpret_cast<float*>(B_(grad_key)->dev);
    p.dv = reinterpret_cast<float*>(B_(grad_value)->dev);
    cudaError_t e = launch_bwd_dkv_only(p, st);
    if (e != cudaSuccess) return cuda_fail(e, "dkv launch");
    sync.out(B_(grad_key)); sync.out(B_(grad_value));
    if ((e = sync.finish()) != cudaSuccess) return cuda_fail(e, "dkv sync");
    return MFA_SUCCESS;
  }
  BwdArgs a{B_(grad_output), B_(q), B_(k), B_(v), outb, B_(logsumexp), B_(grad_query), nullptr, nullptr, B_(d_values),
            B, Sq, Skv, H, Hkv, D, scale, causal, -1, dt, kF32, false, false, false, false,
            MaskArgs{nullptr, 0, nullptr, nullptr, 0, 0, 0}, qv(q_scale, q_zp, qbs, qblk), qv(k_scale, k_zp, kbs, kblk),
            qv(v_scale, v_zp, vbs, vblk), nullptr, false, true, false};
  return backward_core(ctx, a);
}

int32_t mfa_attention_backward_query_quantized(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t output,
    mfa_buffer_t grad_output, mfa_buffer_t logsumexp, mfa_buffer_t grad_query, mfa_buffer_t d_values,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    int32_t q_precision, int32_t k_precision, int32_t v_precision, bool causal, bool, bool, bool, bool) {
  return prequantised_backward(context, q, k, v, output, grad_output, logsumexp, grad_query, nullptr, nullptr, d_values,
                               batch_size, seq_len_q, seq_len_kv, num_heads, num_heads, head_dim, q_scale, q_zero_point,
                               k_scale, k_zero_point, v_scale, v_zero_point, q_precision, k_precision, v_precision,
                               causal, true, nullptr, nullptr, nullptr, 0, 0, 0);
}

int32_t mfa_attention_backward_kv_quantized(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v,
    mfa_buffer_t grad_output, mfa_buffer_t logsumexp, mfa_buffer_t d_values,
    mfa_buffer_t grad_key, mfa_buffer_t grad_value,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    int32_t q_precision, int32_t k_precision, int32_t v_precision, bool causal, bool, bool, bool, bool) {
  return prequantised_backward(context, q, k, v, nullptr, grad_output, logsumexp, nullptr, grad_key, grad_value, d_values,
                               batch_size, seq_len_q, seq_len_kv, num_heads, num_heads, head_dim, q_scale, q_zero_point,
                               k_scale, k_zero_point, v_scale, v_zero_point, q_precision, k_precision, v_precision,
                               causal, false, nullptr, nullptr, nullptr, 0, 0, 0);
}

int32_t mfa_attention_backward_query_quantized_ex(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t output,
    mfa_buffer_t grad_output, mfa_buffer_t logsumexp, mfa_buffer_t grad_query, mfa_buffer_t d_values,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint32_t num_kv_heads,
    uint16_t head_dim,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    int32_t q_precision, int32_t k_precision, int32_t v_precision, bool causal, bool, bool, bool, bool,
    mfa_buffer_t q_block_scales, mfa_buffer_t, mfa_buffer_t k_block_scales, mfa_buffer_t,
    mfa_buffer_t v_block_scales, mfa_buffer_t,
    uint32_t q_block_size, uint32_t k_block_size, uint32_t v_block_size, uint32_t) {
  return prequantised_backward(context, q, k, v, output, grad_output, logsumexp, grad_query, nullptr, nullptr, d_values,
                               batch_size, seq_len_q, seq_len_kv, num_heads, num_kv_heads ? num_kv_heads : num_heads,
                               head_dim, q_scale, q_zero_point, k_scale, k_zero_point, v_scale, v_zero_point,
                               q_precision, k_precision, v_precision, causal, true, q_block_scales, k_block_scales,
                               v_block_scales, q_block_size, k_block_size, v_block_size);
}

int32_t mfa_attention_backward_kv_quantized_ex(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v,
    mfa_buffer_t grad_output, mfa_buffer_t logsumexp, mfa_buffer_t d_values,
    mfa_buffer_t grad_key, mfa_buffer_t grad_value,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint32_t num_kv_heads,
    uint16_t head_dim,
    float q_scale, int32_t q_zero_point, float k_scale, int32_t k_zero_point, float v_scale, int32_t v_zero_point,
    int32_t q_precision, int32_t k_precision, int32_t v_precision, bool causal, bool, bool, bool, bool,
    mfa_buffer_t q_block_scales, mfa_buffer_t, mfa_buffer_t k_block_scales, mfa_buffer_t,
    mfa_buffer_t v_block_scales, mfa_buffer_t,
    uint32_t q_block_size, uint32_t k_block_size, uint32_t v_block_size, uint32_t) {
  return prequantised_backward(context, q, k, v, nullptr, grad_output, logsumexp, nullptr, grad_key, grad_value, d_values,
                               batch_size, seq_len_q, seq_len_kv, num_heads, num_kv_heads ? num_kv_heads : num_heads,
                               head_dim, q_scale, q_zero_point, k_scale, k_zero_point, v_scale, v_zero_point,
                               q_precision, k_precision, v_precision, causal, false, q_block_scales, k_block_scales,
                               v_block_scales, q_block_size, k_block_size, v_block_size);
}

int32_t mfa_quantized_backward(
    mfa_context_t context, mfa_buffer_t q, mfa_buffer_t k, mfa_buffer_t v, mfa_buffer_t out,
    mfa_buffer_t grad_out, mfa_buffer_t lse, mfa_buffer_t grad_q, mfa_buffer_t grad_k, mfa_buffer_t grad_v,
    mfa_buffer_t mask,
    uint32_t batch_size, uint32_t seq_len_q, uint32_t seq_len_kv, uint32_t num_heads, uint16_t head_dim,
    float softmax_scale, bool causal, int32_t target_precision, int32_t quant_mode, int32_t input_precision) {
  if (!context || !q || !k || !v || !out || !grad_out || !lse || !grad_q || !grad_k || !grad_v) return MFA_ERROR_INVALID_ARGS;
  const int in_dt = header_precision_to_dtype(input_precision);
  if (!valid_float_dtype(in_dt)) return MFA_ERROR_INVALID_ARGS;
  if (target_precision != MFA_PRECISION_INT8 && target_precision != MFA_PRECISION_INT4) return MFA_ERROR_INVALID_ARGS;
  if (quant_mode != 0 && quant_mode != 2) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  Context* ctx = C_(context);
  const uint32_t B = batch_size, H = num_heads, Sq = seq_len_q, Skv = seq_len_kv, D = head_dim;
  const uint32_t blk = quant_mode == 2 ? 64 : 0;
  if (mask && B_(mask)->bytes < (size_t)B * H * Sq * Skv * 4) return MFA_ERROR_INVALID_ARGS;
  // Re-quantise Q, K, V exactly as the forward did (deterministic), then run the backward on the codes.  The context lock
  // (recursive) and the scratch scope are held across BOTH phases: no other call can overwrite the codes or scales between
  // the quantise kernels and the backward kernels that read them.
  QuantView qq, qk, qvv;
  TensorView tq, tk, tv;
  int d0, d1, d2;
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  cudaStream_t st = ctx->stream;
  ScratchScope scope(ctx, st);
  {
    Sync sync{ctx, st, false, {}};
    cudaError_t e;
    if ((e = sync.in(B_(q))) != cudaSuccess || (e = sync.in(B_(k))) != cudaSuccess || (e = sync.in(B_(v))) != cudaSuccess ||
        (e = sync.in(B_(mask))) != cudaSuccess)
      return cuda_fail(e, "h2d");
    mfa_error_t me;
    QOperand oq{B_(q), in_dt, 1.f, 0, blk}, ok{B_(k), in_dt, 1.f, 0, blk}, ov{B_(v), in_dt, 1.f, 0, blk};
    if ((me = quantise_operand(scope, st, oq, 0, B, H, Sq, D, target_precision, tq, qq, d0)) != MFA_SUCCESS) return me;
    if ((me = quantise_operand(scope, st, ok, 1, B, H, Skv, D, target_precision, tk, qk, d1)) != MFA_SUCCESS) return me;
    if ((me = quantise_operand(scope, st, ov, 2, B, H, Skv, D, target_precision, tv, qvv, d2)) != MFA_SUCCESS) return me;
  }
  // Wrap the device-resident codes as transient buffers and reuse backward_core (stream order keeps the
  // quantise kernels ahead of the backward kernels).
  Buffer cq, ck, cv;
  cq.dev = const_cast<void*>(tq.ptr); cq.bytes = packed_bytes(elems(B, H, Sq, D), d0);
  ck.dev = const_cast<void*>(tk.ptr); ck.bytes = packed_bytes(elems(B, H, Skv, D), d1);
  cv.dev = const_cast<void*>(tv.ptr); cv.bytes = packed_bytes(elems(B, H, Skv, D), d2);
  MaskArgs m{nullptr, 0, nullptr, nullptr, 0, 0, 0};
  int64_t mshape[4] = {B, H, Sq, Skv}, mstr[4] = {(int64_t)H * Sq * Skv, (int64_t)Sq * Skv, Skv, 1};
  if (mask) m = MaskArgs{B_(mask)->dev, B_(mask)->bytes, mshape, mstr, 4, MFA_MASK_TYPE_ADDITIVE, MFA_MASK_SCALAR_FP32};
  BwdArgs a{B_(grad_out), &cq, &ck, &cv, B_(out), B_(lse), B_(grad_q), B_(grad_k), B_(grad_v), nullptr,
            B, Sq, Skv, H, H, D, softmax_scale, causal, -1, d0, kF32, false, false, false, false, m, qq, qk, qvv,
            nullptr, false, true, true};
  return backward_core(ctx, a);
}

// ---- misc -------------------------------------------------------------------------------------------------
mfa_error_t mfa_sparse_indexer_scores(mfa_context_t, mfa_buffer_t, mfa_buffer_t, uint32_t, uint32_t, uint32_t, uint32_t,
                                      uint16_t, float, mfa_buffer_t, mfa_buffer_t*) {
  return MFA_ERROR_DEVICE_NOT_SUPPORTED;   // out of the hot path (SURVEY section 2 row 13)
}

const char* mfa_error_string(mfa_error_t error) {
  const char* s = (error >= 0 && error <= 5) ? kErrStr[error] : "Unknown error";
  return strdup(s);
}

bool mfa_is_device_supported(void) { return device_ok(); }

void mfa_get_version(int* major, int* minor, int* patch) {
  if (major) *major = 1;
  if (minor) *minor = 0;
  if (patch) *patch = 0;
}

double mfa_get_gpu_latency(mfa_context_t context) { return context ? C_(context)->last_latency : 0.0; }

mfa_error_t mfa_set_scale_arrays(mfa_context_t context, const float* q_scales, uint32_t nq, const float* k_scales,
                                 uint32_t nk, const float* v_scales, uint32_t nv) {
  if (!context) return MFA_ERROR_INVALID_ARGS;
  Context* ctx = C_(context);
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  const float* src[3] = {q_scales, k_scales, v_scales};
  const uint32_t n[3] = {nq, nk, nv};
  for (int i = 0; i < 3; ++i) {
    if (src[i] && n[i]) ctx->row_scales[i].assign(src[i], src[i] + n[i]);
    else ctx->row_scales[i].clear();
  }
  return MFA_SUCCESS;
}

int32_t mfa_has_native_bfloat(void) { return device_ok() ? 1 : 0; }
int32_t mfa_has_native_bfloat_msl32(void) { return device_ok() ? 1 : 0; }

int32_t mfa_hadamard_rotate(mfa_buffer_t data, uint32_t block_size, uint32_t num_blocks) {
  if (!data) return MFA_ERROR_INVALID_ARGS;
  if (block_size == 0 || block_size > 1024 || (block_size & (block_size - 1))) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  Buffer* b = B_(data);
  if (b->bytes < (size_t)block_size * num_blocks * 4) return MFA_ERROR_INVALID_ARGS;
  Context* ctx = b->owner;                         // no context argument in the reference ABI: the buffer knows its context
  {
    std::lock_guard<std::mutex> glock(g_ctx_mu);
    bool alive = false;
    for (int i = 0; i < kMaxDevices; ++i) alive |= g_ctxs[i] != nullptr && g_ctxs[i] == ctx;
    if (!alive) return MFA_ERROR_INVALID_ARGS;      // buffers only exist under a live context
  }
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  Sync sync{ctx, ctx->stream, false, {}};
  cudaError_t e = sync.in(b);
  if (e == cudaSuccess) e = launch_hadamard(reinterpret_cast<float*>(b->dev), block_size, num_blocks, ctx->stream);
  if (e != cudaSuccess) return cuda_fail(e, "hadamard");
  sync.out(b);
  return sync.finish() == cudaSuccess ? MFA_SUCCESS : MFA_ERROR_EXECUTION_FAILED;
}

int mfa_rope_rotate_encode_mtl(
    mfa_context_t context, void* command_buffer,
    void* src, int64_t src_offset, int64_t sB, int64_t sH, int64_t sS,
    void* dst, int64_t dst_offset, void* cos_table, int64_t cos_offset, void* sin_table, int64_t sin_offset,
    int64_t table_batch_stride, bool negate_sin, uint32_t B, uint32_t H, uint32_t S, uint32_t D, const char* precision) {
  if (!context || !src || !dst || !cos_table || !sin_table) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  const int dt = parse_precision_str(precision);
  if (!valid_float_dtype(dt) || (D & 1)) return MFA_ERROR_INVALID_ARGS;
  Context* ctx = C_(context);
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  cudaError_t e = launch_rope(reinterpret_cast<char*>(src) + src_offset, reinterpret_cast<char*>(dst) + dst_offset,
                              reinterpret_cast<const float*>(reinterpret_cast<char*>(cos_table) + cos_offset),
                              reinterpret_cast<const float*>(reinterpret_cast<char*>(sin_table) + sin_offset), sB, sH, sS,
                              table_batch_stride, negate_sin, B, H, S, D, dt, reinterpret_cast<cudaStream_t>(command_buffer));
  return e == cudaSuccess ? MFA_SUCCESS : cuda_fail(e, "rope");
}

mfa_error_t mfa_quantize(mfa_context_t context, mfa_buffer_t src, mfa_buffer_t codes, mfa_buffer_t scales, uint64_t rows,
                         uint64_t cols, uint32_t block_rows, uint32_t block_cols, mfa_precision_t src_precision,
                         mfa_precision_t target_precision, float scale_floor, void* stream) {
  if (!context || !src || !codes || !scales) return MFA_ERROR_INVALID_ARGS;
  const int sdt = header_precision_to_dtype(src_precision);
  if (!valid_float_dtype(sdt)) return MFA_ERROR_INVALID_ARGS;
  if (target_precision != MFA_PRECISION_INT8 && target_precision != MFA_PRECISION_INT4) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  const int bits = target_precision == MFA_PRECISION_INT8 ? 8 : 4;
  const uint64_t n = rows * cols;
  const uint64_t br = (block_rows == 0 || block_rows > rows) ? rows : block_rows;
  const uint64_t bc = (block_cols == 0 || block_cols > cols) ? cols : block_cols;
  const uint64_t nb = n ? ((rows + br - 1) / br) * ((cols + bc - 1) / bc) : 0;
  Buffer *bs = B_(src), *bcodes = B_(codes), *bsc = B_(scales);
  if (bs->bytes < n * dtype_bytes(sdt) || bcodes->bytes < (bits == 8 ? n : (n + 1) / 2) || bsc->bytes < nb * 4)
    return MFA_ERROR_INVALID_ARGS;
  const bool async = stream != nullptr;
  if (async && (bs->mirrored || bcodes->mirrored || bsc->mirrored)) return MFA_ERROR_INVALID_ARGS;
  Context* ctx = C_(context);
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  cudaStream_t st = async ? reinterpret_cast<cudaStream_t>(stream) : ctx->stream;
  Sync sync{ctx, st, async, {}};
  cudaError_t e = sync.in(bs);
  if (e != cudaSuccess) return cuda_fail(e, "h2d");
  Timer tm(ctx, st, !async);
  e = launch_quantize(bs->dev, sdt, bcodes->dev, reinterpret_cast<float*>(bsc->dev), rows, cols, block_rows, block_cols,
                      bits, scale_floor, st);
  tm.stop();
  ctx->last_kernel = g_last_kernel;
  if (e == cudaErrorInvalidValue) { cudaGetLastError(); return MFA_ERROR_INVALID_ARGS; }
  if (e != cudaSuccess) return cuda_fail(e, "quantize");
  sync.out(bcodes); sync.out(bsc);
  if ((e = sync.finish()) != cudaSuccess) return cuda_fail(e, "quantize sync");
  tm.read();
  return MFA_SUCCESS;
}

mfa_error_t mfa_dequantize(mfa_context_t context, mfa_buffer_t codes, mfa_buffer_t scales, mfa_buffer_t out, uint64_t rows,
                           uint64_t cols, uint32_t block_rows, uint32_t block_cols, mfa_precision_t code_precision,
                           void* stream) {
  if (!context || !codes || !scales || !out) return MFA_ERROR_INVALID_ARGS;
  if (code_precision != MFA_PRECISION_INT8 && code_precision != MFA_PRECISION_INT4) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  const int bits = code_precision == MFA_PRECISION_INT8 ? 8 : 4;
  const uint64_t n = rows * cols;
  Buffer *bcodes = B_(codes), *bsc = B_(scales), *bo = B_(out);
  if (bcodes->bytes < (bits == 8 ? n : (n + 1) / 2) || bo->bytes < n * 4) return MFA_ERROR_INVALID_ARGS;
  {
    const uint64_t br = (block_rows == 0 || block_rows > rows) ? rows : block_rows;
    const uint64_t bc = (block_cols == 0 || block_cols > cols) ? cols : block_cols;
    const uint64_t nb = n ? ((rows + br - 1) / br) * ((cols + bc - 1) / bc) : 0;
    if (bsc->bytes < nb * 4) return MFA_ERROR_INVALID_ARGS;
  }
  const bool async = stream != nullptr;
  if (async && (bo->mirrored || bcodes->mirrored || bsc->mirrored)) return MFA_ERROR_INVALID_ARGS;
  Context* ctx = C_(context);
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  cudaStream_t st = async ? reinterpret_cast<cudaStream_t>(stream) : ctx->stream;
  Sync sync{ctx, st, async, {}};
  cudaError_t e;
  if ((e = sync.in(bcodes)) != cudaSuccess || (e = sync.in(bsc)) != cudaSuccess) return cuda_fail(e, "h2d");
  e = launch_dequantize(bcodes->dev, reinterpret_cast<const float*>(bsc->dev), reinterpret_cast<float*>(bo->dev), rows,
                        cols, block_rows, block_cols, bits, st);
  if (e != cudaSuccess) return cuda_fail(e, "dequantize");
  sync.out(bo);
  return sync.finish() == cudaSuccess ? MFA_SUCCESS : MFA_ERROR_EXECUTION_FAILED;
}

mfa_error_t mfa_merge_partials(mfa_context_t context, mfa_buffer_t o_acc, mfa_buffer_t l_acc, mfa_buffer_t o_part,
                               mfa_buffer_t l_part, uint64_t rows, uint32_t head_dim, void* stream) {
  if (!context || !o_acc || !l_acc || !o_part || !l_part) return MFA_ERROR_INVALID_ARGS;
  if (!device_ok()) return MFA_ERROR_DEVICE_NOT_SUPPORTED;
  Buffer* bs[4] = {B_(o_acc), B_(l_acc), B_(o_part), B_(l_part)};
  if (bs[0]->bytes < rows * head_dim * 4 || bs[2]->bytes < rows * head_dim * 4 || bs[1]->bytes < rows * 4 ||
      bs[3]->bytes < rows * 4)
    return MFA_ERROR_INVALID_ARGS;
  const bool async = stream != nullptr;
  for (Buffer* b : bs) if (async && b->mirrored) return MFA_ERROR_INVALID_ARGS;
  Context* ctx = C_(context);
  std::lock_guard<std::recursive_mutex> lock(ctx->mu);
  DeviceGuard dg(ctx->device);
  cudaStream_t st = async ? reinterpret_cast<cudaStream_t>(stream) : ctx->stream;
  Sync sync{ctx, st, async, {}};
  for (Buffer* b : bs) { cudaError_t e = sync.in(b); if (e != cudaSuccess) return cuda_fail(e, "h2d"); }
  cudaError_t e = launch_merge_partials(reinterpret_cast<float*>(bs[0]->dev), reinterpret_cast<float*>(bs[1]->dev),
                                        reinterpret_cast<const float*>(bs[2]->dev),
                                        reinterpret_cast<const float*>(bs[3]->dev), rows, head_dim, st);
  if (e != cudaSuccess) return cuda_fail(e, "merge");
  sync.out(bs[0]); sync.out(bs[1]);
  return sync.finish() == cudaSuccess ? MFA_SUCCESS : MFA_ERROR_EXECUTION_FAILED;
}

mfa_error_t mfa_set_quantized_pv_precision(mfa_context_t context, int32_t precision) {
  if (!context) return MFA_ERROR_INVALID_ARGS;
  if (precision != MFA_PRECISION_BF16 && precision != MFA_PRECISION_FP8_E4M3) return MFA_ERROR_INVALID_ARGS;
  std::lock_guard<std::recursive_mutex> lock(C_(context)->mu);
  fwd_tcq_set_pv_mode(precision == MFA_PRECISION_BF16);
  return MFA_SUCCESS;
}

int32_t mfa_get_quantized_pv_precision(mfa_context_t) { return fwd_tcq_pv_mode() == 1 ? MFA_PRECISION_BF16 : MFA_PRECISION_FP8_E4M3; }

const char* mfa_last_kernel_name(mfa_context_t context) { return context ? C_(context)->last_kernel : "none"; }
uint64_t mfa_launch_count(mfa_context_t) { return g_launch_count; }

// ---- MLA: outside the attention hot path (SURVEY section 2 row 9) -------------------------------------------
mfa_error_t mfa_mla_create_context(mfa_mla_context_t* context) {
  if (!context) return MFA_ERROR_INVALID_ARGS;
  *context = malloc(8);
  return *context ? MFA_SUCCESS : MFA_ERROR_MEMORY_ALLOCATION;
}
void mfa_mla_destroy_context(mfa_mla_context_t context) { free(context); }
mfa_error_t mfa_mla_init_weights(mfa_mla_context_t, uint32_t, uint32_t, uint32_t) { return MFA_ERROR_DEVICE_NOT_SUPPORTED; }
mfa_error_t mfa_mla_load_weights(mfa_mla_context_t, mfa_buffer_t, mfa_buffer_t) { return MFA_ERROR_DEVICE_NOT_SUPPORTED; }
mfa_error_t mfa_mla_forward(mfa_mla_context_t, mfa_context_t, mfa_buffer_t, mfa_buffer_t*, mfa_buffer_t*, uint32_t, uint32_t,
                            uint32_t, uint32_t, uint32_t) {
  return MFA_ERROR_DEVICE_NOT_SUPPORTED;
}

}  // extern "C"
