// capi.cu -- the C ABI of libcodexcommit.so (include/codex_commit.h) over the sm_100a kernels.
// No CPU arithmetic lives here: every field operation is a kernel launch; without a CUDA device the context
// cannot be created and every entry point fails.
#include "../../include/codex_commit.h"

#include <cuda_runtime.h>

#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <new>
#include <thread>
#include <unordered_map>
#include <vector>

#include "kernels.cuh"
#include "slot_builder.h"
#include "slot_image.h"

using namespace cdx;

// ---------------------------------------------------------------------------------------------------------

#define CDX_MAX_STAGE 4

struct cdx_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;       // compute
  cudaStream_t copy_stream = nullptr;  // H2D staging for *_host entry points
  cudaStream_t copy_stream2 = nullptr; // second H2D stream: the copies of consecutive tiles of a pinned slot alternate (two in flight)
  cudaStream_t stream2 = nullptr;      // second compute stream: odd tiles of a streamed slot (kernels overlap at the tile seams)
  cudaEvent_t ev_join = nullptr;
  cudaEvent_t ev_copied[CDX_MAX_STAGE] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_consumed[CDX_MAX_STAGE] = {nullptr, nullptr, nullptr, nullptr};
  void* d_stage[CDX_MAX_STAGE] = {nullptr, nullptr, nullptr, nullptr};   // device tiles the non-resident pipelines stream through
  size_t stage_bytes = 0;
  int stage_count = 0;
  int stage_tiles = 3;                 // tiles in flight for pinned host slots (CODEX_COMMIT_STAGE_TILES = 2..4)
  size_t tile_mib = 256;               // tile size of the non-resident pipelines (CODEX_COMMIT_TILE_MIB)
  int ramp_mode = 2;                   // how a pinned host slot's pipeline starts (CODEX_COMMIT_RAMP = 0, 1 or 2 = auto; see hash_cells_pinned)
  cudaEvent_t ev_rate[2] = {nullptr, nullptr};   // around one full-size tile copy of the last pinned commit: the H2D rate this GPU really gets
  size_t rate_bytes = 0;
  double h2d_gbs = 0.0;                // last measured rate (0 = not measured yet)
  void* h_pinned[2] = {nullptr, nullptr};   // pinned read buffers of cdx_slot_commit_file
  size_t pinned_bytes = 0;
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr};
  void* h_scratch = nullptr;           // small pinned buffer for per-call tables uploaded without stalling a busy stream (batch offsets)
  size_t scratch_bytes = 0;
  cudaEvent_t ev_scratch = nullptr;    // recorded after the last upload from h_scratch
  uint64_t launches = 0;
  bool no_bounce = false;              // CODEX_COMMIT_NO_BOUNCE=1: pageable host slots straight through cudaMemcpyAsync (A/B only)
  bool tma_smem_set = false;
  size_t max_launch_cells = (size_t)1 << 30;   // cells per cell-sponge launch (CODEX_COMMIT_MAX_LAUNCH_CELLS lowers it so tests can cross the boundary)
  bool plain_loads = false;            // CODEX_COMMIT_PLAIN_LOADS=1: per-thread global loads instead of the TMA-staged rows (A/B only)
  char err[256] = {0};
};

struct cdx_slot {
  cdx_ctx* ctx = nullptr;
  cudaStream_t stream = nullptr;
  size_t cell_size = 0, block_size = 0;
  uint64_t n_local_cells = 0, n_local_blocks = 0, first_block = 0, n_total_blocks = 0;
  uint32_t cpb_log2 = 0;        // log2(cells per block)
  uint32_t block_depth = 0;     // path levels inside a block tree (= cpb_log2, or 1 for one-cell blocks)
  uint32_t slot_depth = 0;      // layers-1 of the slot tree
  uint32_t top_level = 0;       // levels < top_level are held for the local range only
  bool has_top = false;
  uint8_t* d_forest = nullptr;  // block-forest levels 0..block_depth, concatenated
  uint8_t* d_low = nullptr;     // slot levels 1..top_level (local ranges), concatenated
  uint8_t* d_top = nullptr;     // slot levels top_level..slot_depth (global), concatenated
  bool top0_alias = false;      // top level storage for level top_level aliases forest/low (non-sharded case)
  bool compact = false;         // cdx_slot_compact: d_forest holds only the block hashes, forest[l < block_depth] are null
  std::vector<uint8_t*> forest, low, top;             // per-level pointers (low[0] aliases forest[block_depth])
  std::vector<uint64_t> low_first, low_count, width;  // width[l] = global width of slot level l
};

namespace {   // device allocations between optional guard bands (defined below, CODEX_COMMIT_GUARD)
bool guard_enabled();
void dev_free(void* p, cudaStream_t st);
}  // namespace

static int fail(cdx_ctx* ctx, int status, const char* fmt, ...) {
  if (ctx) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(ctx->err, sizeof ctx->err, fmt, ap);
    va_end(ap);
  }
  return status;
}

#define CU_TRY(ctx, call)                                                                         \
  do {                                                                                            \
    cudaError_t _e = (call);                                                                      \
    if (_e != cudaSuccess)                                                                        \
      return fail((ctx), CDX_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

static inline unsigned grid_for(size_t n, unsigned block = CDX_BLOCK) { return (unsigned)((n + block - 1) / block); }

// CTA width for a launch of n threads: the compiled width when the launch fills the machine, narrower CTAs (down to one
// warp) when it does not, so that a small launch -- a 4 MiB slot is 2048 cells, the upper tree levels a handful of nodes --
// spreads over as many SMs as it has warps.  Every thread of these kernels runs a long dependent chain of
// multiplications; two warps sharing an SM sub-partition finish later than two warps on two SMs.
static inline unsigned block_for(const cdx_ctx* ctx, size_t n) {
  unsigned b = CDX_BLOCK;
  while (b > 32 && n < (size_t)ctx->sm_count * b) b >>= 1;
  return b;
}

#define LAUNCH(ctx, kernel, n_threads, stream, ...)                                    \
  do {                                                                                 \
    const unsigned _b = block_for((ctx), (n_threads));                                 \
    kernel<<<grid_for((n_threads), _b), _b, 0, (stream)>>>(__VA_ARGS__);               \
    (ctx)->launches++;                                                                 \
    CU_TRY(ctx, cudaGetLastError());                                                   \
  } while (0)

// ---- context ------------------------------------------------------------------------------------------------

extern "C" int cdx_abi_version(void) { return CDX_ABI_VERSION; }

extern "C" int cdx_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

extern "C" const char* cdx_status_string(int s) {
  switch (s) {
    case CDX_OK: return "ok";
    case CDX_ERR_ARG: return "bad argument";
    case CDX_ERR_SIZE: return "sizes are not divisible as required";
    case CDX_ERR_NOT_POW2: return "number of cells must be a power of two";
    case CDX_ERR_RANGE: return "index or depth out of range";
    case CDX_ERR_CUDA: return "CUDA error / no device";
    case CDX_ERR_ALLOC: return "allocation failed";
    case CDX_ERR_STATE: return "handle is not in the required state";
    case CDX_ERR_MISMATCH: return "slot bytes do not match the commitment";
    default: return "unknown status";
  }
}

extern "C" int cdx_ctx_create(int device, cdx_ctx** out) {
  if (!out) return CDX_ERR_ARG;
  *out = nullptr;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0 || device < 0 || device >= n_dev) return CDX_ERR_CUDA;
  cdx_ctx* ctx = new (std::nothrow) cdx_ctx();
  if (!ctx) return CDX_ERR_ALLOC;
  ctx->device = device;
  if (const char* v = getenv("CODEX_COMMIT_PLAIN_LOADS")) ctx->plain_loads = v[0] == '1';
  if (const char* v = getenv("CODEX_COMMIT_NO_BOUNCE")) ctx->no_bounce = v[0] == '1';
  if (const char* v = getenv("CODEX_COMMIT_MAX_LAUNCH_CELLS")) {
    const long long n = atoll(v);
    if (n >= 32 && n <= (1ll << 30)) ctx->max_launch_cells = (size_t)n & ~(size_t)31;   // whole warps
  }
  if (const char* v = getenv("CODEX_COMMIT_STAGE_TILES")) {
    const int n = atoi(v);
    if (n >= 2 && n <= CDX_MAX_STAGE) ctx->stage_tiles = n;
  }
  if (const char* v = getenv("CODEX_COMMIT_RAMP")) ctx->ramp_mode = v[0] == '0' ? 0 : (v[0] == '1' ? 1 : 2);
  if (const char* v = getenv("CODEX_COMMIT_TILE_MIB")) {
    const long n = atol(v);
    if (n >= 16 && n <= 4096) ctx->tile_mib = (size_t)n;
  }
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
  if (e == cudaSuccess) {   // keep freed tree buffers in the pool instead of returning them to the driver
    cudaMemPool_t pool;
    e = cudaDeviceGetDefaultMemPool(&pool, device);
    if (e == cudaSuccess) {
      uint64_t never = UINT64_MAX;
      e = cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &never);
    }
  }
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_stream2, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_scratch, cudaEventDisableTiming);
  for (int i = 0; i < CDX_MAX_STAGE && e == cudaSuccess; ++i) {
    e = cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_consumed[i], cudaEventDisableTiming);
  }
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&ctx->ev_h2d[i], cudaEventDisableTiming);
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaEventCreate(&ctx->ev_rate[i]);
  if (e != cudaSuccess) {
    delete ctx;
    return CDX_ERR_CUDA;
  }
  *out = ctx;
  return CDX_OK;
}

// The staging ring comes from cudaMalloc, not from the stream-ordered pool: without guard bands it goes back through cudaFree.
static void release_stage(cdx_ctx* ctx) {
  for (int i = 0; i < CDX_MAX_STAGE; ++i) {
    if (ctx->d_stage[i]) {
      if (guard_enabled()) dev_free(ctx->d_stage[i], ctx->stream);
      else cudaFree(ctx->d_stage[i]);
    }
    ctx->d_stage[i] = nullptr;
  }
  ctx->stage_bytes = 0;
  ctx->stage_count = 0;
}

extern "C" void cdx_ctx_destroy(cdx_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  release_stage(ctx);
  for (int i = 0; i < CDX_MAX_STAGE; ++i) {
    if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]);
    if (ctx->ev_consumed[i]) cudaEventDestroy(ctx->ev_consumed[i]);
  }
  for (int i = 0; i < 2; ++i) {
    if (ctx->h_pinned[i]) cudaFreeHost(ctx->h_pinned[i]);
    if (ctx->ev_h2d[i]) cudaEventDestroy(ctx->ev_h2d[i]);
    if (ctx->ev_rate[i]) cudaEventDestroy(ctx->ev_rate[i]);
  }
  if (ctx->copy_stream2) cudaStreamDestroy(ctx->copy_stream2);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->ev_scratch) cudaEventDestroy(ctx->ev_scratch);
  if (ctx->h_scratch) cudaFreeHost(ctx->h_scratch);
  delete ctx;
}

extern "C" const char* cdx_last_error(const cdx_ctx* ctx) { return ctx ? ctx->err : "no context"; }
extern "C" uint64_t cdx_launch_count(const cdx_ctx* ctx) { return ctx ? ctx->launches : 0; }
extern "C" void* cdx_ctx_stream(const cdx_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

// ---- device allocations, optionally between guard bands -------------------------------------------------------------
// compute-sanitizer is not available on the GPU pool this library is developed on.  CODEX_COMMIT_GUARD=1 is the
// substitute for out-of-bounds WRITES: every device allocation of the library (tree layers, staging tiles, scoped
// buffers) gets a 4 KiB band of 0xA5 on either side, and freeing it first reads the bands back; a damaged band is
// reported on stderr and aborts the process.  A debug mode: the check synchronises the stream at every free.
namespace {
constexpr size_t kGuardBytes = 4096;
struct GuardInfo {
  size_t bytes;
  bool stream_ordered;
};
bool guard_enabled() {
  static const bool on = [] {
    const char* v = getenv("CODEX_COMMIT_GUARD");
    return v && v[0] == '1';
  }();
  return on;
}
std::mutex g_guard_mutex;
std::unordered_map<void*, GuardInfo> g_guard_live;

cudaError_t dev_alloc(void** p, size_t bytes, cudaStream_t st, bool stream_ordered = true) {
  if (bytes == 0) bytes = 1;
  if (!guard_enabled()) return stream_ordered ? cudaMallocAsync(p, bytes, st) : cudaMalloc(p, bytes);
  uint8_t* raw = nullptr;
  const size_t padded = (bytes + 255) / 256 * 256;       // the far band starts 256-byte aligned as well
  cudaError_t e = stream_ordered ? cudaMallocAsync((void**)&raw, padded + 2 * kGuardBytes, st) : cudaMalloc((void**)&raw, padded + 2 * kGuardBytes);
  if (e != cudaSuccess) return e;
  e = cudaMemsetAsync(raw, 0xA5, kGuardBytes, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(raw + kGuardBytes + bytes, 0xA5, padded - bytes + kGuardBytes, st);
  if (e != cudaSuccess) return e;
  *p = raw + kGuardBytes;
  std::lock_guard<std::mutex> lock(g_guard_mutex);
  g_guard_live[*p] = GuardInfo{bytes, stream_ordered};
  return cudaSuccess;
}

void dev_free(void* p, cudaStream_t st) {
  if (!p) return;
  if (!guard_enabled()) {
    cudaFreeAsync(p, st);
    return;
  }
  GuardInfo info{0, true};
  {
    std::lock_guard<std::mutex> lock(g_guard_mutex);
    auto it = g_guard_live.find(p);
    if (it == g_guard_live.end()) {
      fprintf(stderr, "CODEX_COMMIT_GUARD: free of an unknown device pointer %p\n", p);
      abort();
    }
    info = it->second;
    g_guard_live.erase(it);
  }
  uint8_t* raw = (uint8_t*)p - kGuardBytes;
  const size_t padded = (info.bytes + 255) / 256 * 256, tail = padded - info.bytes + kGuardBytes;
  std::vector<uint8_t> head(kGuardBytes), far(tail);
  cudaMemcpyAsync(head.data(), raw, kGuardBytes, cudaMemcpyDeviceToHost, st);
  cudaMemcpyAsync(far.data(), raw + kGuardBytes + info.bytes, tail, cudaMemcpyDeviceToHost, st);
  if (cudaStreamSynchronize(st) != cudaSuccess) cudaGetLastError();
  for (size_t i = 0; i < kGuardBytes; ++i)
    if (head[i] != 0xA5) {
      fprintf(stderr, "CODEX_COMMIT_GUARD: %zu-byte allocation %p: write %zu bytes BEFORE its start\n", info.bytes, p, kGuardBytes - i);
      abort();
    }
  for (size_t i = 0; i < tail; ++i)
    if (far[i] != 0xA5) {
      fprintf(stderr, "CODEX_COMMIT_GUARD: %zu-byte allocation %p: write %zu bytes PAST its end\n", info.bytes, p, i);
      abort();
    }
  if (info.stream_ordered) cudaFreeAsync(raw, st);
  else cudaFree(raw);
}
}  // namespace

// Scoped device buffer for the *_host entry points.  Stream-ordered allocation from the device's default memory
// pool (release threshold raised to "never" in cdx_ctx_create): cudaMalloc/cudaFree cost tens to hundreds of
// milliseconds for tree-sized buffers on this platform and serialise the device, cudaMallocAsync/cudaFreeAsync
// reuse pooled memory in microseconds.
struct DevBuf {
  void* p = nullptr;
  cudaStream_t st = nullptr;
  ~DevBuf() {
    if (p) dev_free(p, st);
  }
  cudaError_t alloc(size_t bytes, cudaStream_t stream) {
    st = stream;
    return dev_alloc(&p, bytes, stream);
  }
  uint8_t* u8() const { return static_cast<uint8_t*>(p); }
};

// The cell sponge, with TMA-staged rows whenever the cell geometry allows 32-byte tensor boxes (cell size a multiple of
// 32, 16-byte aligned base, < 2^32 cells); otherwise the same sponge over per-thread global loads.  The tensor map
// is encoded on the host per launch (cuTensorMapEncodeTiled, resolved through the runtime so libcuda is not a link
// dependency) and travels as a __grid_constant__ kernel parameter.
typedef int (*encode_tiled_fn)(void* tensorMap, int dataType, unsigned rank, void* globalAddress, const unsigned long long* globalDim,
                               const unsigned long long* globalStrides, const unsigned* boxDim, const unsigned* elementStrides, int interleave,
                               int swizzle, int l2Promotion, int oobFill);

static encode_tiled_fn get_encode_tiled() {
  static encode_tiled_fn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (encode_tiled_fn)p;
  }
  return fn;
}

// Make a small host table available to kernels on `st` without stalling it: an asynchronous copy from pageable memory
// would first wait for everything queued on the stream, and a copy queued ON the stream would sit behind the sponge that
// runs there.  The device buffer is allocated and filled on the (idle) copy stream from the context's pinned scratch
// buffer, `st` waits for the event, and the buffer is handed over to `st` for its stream-ordered free.  The scratch
// buffer is reused only after the previous upload from it has completed.
static int upload_table(cdx_ctx* ctx, DevBuf& dst, const void* src, size_t bytes, cudaStream_t st) {
  CU_TRY(ctx, cudaEventSynchronize(ctx->ev_scratch));              // never recorded = complete
  if (ctx->scratch_bytes < bytes) {
    if (ctx->h_scratch) cudaFreeHost(ctx->h_scratch);
    ctx->h_scratch = nullptr;
    ctx->scratch_bytes = 0;
    const size_t want = bytes < ((size_t)64 << 10) ? ((size_t)64 << 10) : bytes;
    if (cudaHostAlloc(&ctx->h_scratch, want, cudaHostAllocDefault) != cudaSuccess) return fail(ctx, CDX_ERR_ALLOC, "cudaHostAlloc of %zu bytes failed", want);
    ctx->scratch_bytes = want;
  }
  memcpy(ctx->h_scratch, src, bytes);
  CU_TRY(ctx, dst.alloc(bytes, ctx->copy_stream));
  CU_TRY(ctx, cudaMemcpyAsync(dst.p, ctx->h_scratch, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
  CU_TRY(ctx, cudaEventRecord(ctx->ev_scratch, ctx->copy_stream));
  CU_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_scratch, 0));
  dst.st = st;                                                      // freed after the kernels on st that read it
  return CDX_OK;
}

static int launch_hash_cells(cdx_ctx* ctx, const void* d_data, size_t n_cells, size_t cell_size, uint8_t* d_out, cudaStream_t st) {
  encode_tiled_fn encode = ctx->plain_loads ? nullptr : get_encode_tiled();
  if (encode && cell_size % CDX_SEG_BYTES == 0 && cell_size >= 64 && cell_size < (1u << 31) && (uintptr_t)d_data % 16 == 0) {
    // tensor coordinates are signed 32-bit (a row index >= 2^31 would read as out of bounds, i.e. as zeros): launches of at
    // most 2^30 cells, each with its own tensor-map base
    const size_t max_cells = ctx->max_launch_cells;
    const unsigned blk = block_for(ctx, n_cells);
    const size_t smem_max = 128 + (CDX_BLOCK / 32) * (CDX_RING_SLOTS * CDX_BOX_BYTES + 8 * CDX_RING_SLOTS);
    const size_t smem = 128 + (blk / 32) * (CDX_RING_SLOTS * CDX_BOX_BYTES + 8 * CDX_RING_SLOTS);
    if (smem_max > 48 * 1024 && !ctx->tma_smem_set) {   // per device, once: rings of CTAs wider than 7 warps exceed the default 48 KB
      CU_TRY(ctx, cudaFuncSetAttribute(k_hash_cells_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
      ctx->tma_smem_set = true;
    }
    for (size_t c0 = 0; c0 < n_cells; c0 += max_cells) {
      const size_t nc = n_cells - c0 < max_cells ? n_cells - c0 : max_cells;
      TensorMap2D tmap;
      const unsigned long long dims[2] = {(unsigned long long)cell_size, (unsigned long long)nc};        // innermost first
      const unsigned long long strides[1] = {(unsigned long long)cell_size};                             // bytes between rows
      const unsigned box[2] = {CDX_SEG_BYTES, 32u};
      const unsigned estr[2] = {1u, 1u};
      // CU_TENSOR_MAP_DATA_TYPE_UINT8 = 0, INTERLEAVE_NONE = 0, SWIZZLE_NONE = 0, L2_PROMOTION_NONE = 0, FLOAT_OOB_FILL_NONE = 0 (zeros)
      const int rc = encode(&tmap, 0, 2, (void*)((const uint8_t*)d_data + c0 * cell_size), dims, strides, box, estr, 0, 0, 0, 0);
      if (rc != 0) return fail(ctx, CDX_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", rc);
      k_hash_cells_tma<<<grid_for(nc, blk), blk, smem, st>>>(tmap, nc, (uint32_t)cell_size, d_out + 32 * c0);
      ctx->launches++;
      CU_TRY(ctx, cudaGetLastError());
    }
    return CDX_OK;
  }
  const size_t max_cells = ctx->max_launch_cells;                            // keeps the grid below 2^31 CTAs
  for (size_t c0 = 0; c0 < n_cells; c0 += max_cells) {
    const size_t nc = n_cells - c0 < max_cells ? n_cells - c0 : max_cells;
    const unsigned blk = block_for(ctx, nc);
    k_hash_cells<<<grid_for(nc, blk), blk, 0, st>>>((const uint32_t*)((const uint8_t*)d_data + c0 * cell_size), nc, (uint32_t)(cell_size / 4),
                                                   d_out + 32 * c0);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
  }
  return CDX_OK;
}

// ---- hash layer ---------------------------------------------------------------------------------------------

extern "C" int cdx_permutation_batch_dev(cdx_ctx* ctx, const void* d_in, void* d_out, size_t n, void* stream) {
  if (!ctx || !d_in || !d_out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (n == 0) return CDX_OK;
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  LAUNCH(ctx, k_permutation_batch, n, st, (const uint8_t*)d_in, (uint8_t*)d_out, n);
  return CDX_OK;
}

extern "C" int cdx_permutation_batch_host(cdx_ctx* ctx, const uint8_t* in, uint8_t* out, size_t n) {
  if (!ctx || !in || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (n == 0) return CDX_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf di, dout;
  CU_TRY(ctx, di.alloc(96 * n, ctx->stream));
  CU_TRY(ctx, dout.alloc(96 * n, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(di.p, in, 96 * n, cudaMemcpyHostToDevice, ctx->stream));
  int rc = cdx_permutation_batch_dev(ctx, di.p, dout.p, n, ctx->stream);
  if (rc) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(out, dout.p, 96 * n, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

extern "C" int cdx_sponge_felts_batch_host(cdx_ctx* ctx, const uint8_t* elems, size_t n_items, size_t len, int rate, uint8_t* out) {
  if (!ctx || !out || (!elems && len)) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (rate != 1 && rate != 2) return fail(ctx, CDX_ERR_ARG, "rate must be 1 or 2");
  if (len > 0xffffffffu / 32) return fail(ctx, CDX_ERR_SIZE, "sponge input too long");
  if (n_items == 0) return CDX_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf di, dout;
  CU_TRY(ctx, di.alloc(32 * len * n_items, ctx->stream));
  CU_TRY(ctx, dout.alloc(32 * n_items, ctx->stream));
  if (len) CU_TRY(ctx, cudaMemcpyAsync(di.p, elems, 32 * len * n_items, cudaMemcpyHostToDevice, ctx->stream));
  LAUNCH(ctx, k_sponge_felts, n_items, ctx->stream, di.u8(), n_items, (uint32_t)len, rate, dout.u8());
  CU_TRY(ctx, cudaMemcpyAsync(out, dout.p, 32 * n_items, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

extern "C" int cdx_hash_bytes_batch_host(cdx_ctx* ctx, const uint8_t* data, size_t n_items, size_t len, uint8_t* out) {
  if (!ctx || !out || (!data && len)) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (len > 0x7fffffffu) return fail(ctx, CDX_ERR_SIZE, "byte string too long");
  if (n_items == 0) return CDX_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf di, dout;
  CU_TRY(ctx, di.alloc(len * n_items, ctx->stream));
  CU_TRY(ctx, dout.alloc(32 * n_items, ctx->stream));
  if (len) CU_TRY(ctx, cudaMemcpyAsync(di.p, data, len * n_items, cudaMemcpyHostToDevice, ctx->stream));
  if (len % 4 == 0 && len > 0) {   // pool allocations are 256-byte aligned, so every item is word aligned
    int rc = launch_hash_cells(ctx, di.p, n_items, len, dout.u8(), ctx->stream);
    if (rc) return rc;
  } else {
    LAUNCH(ctx, k_hash_bytes_any, n_items, ctx->stream, di.u8(), n_items, (uint32_t)len, dout.u8());
  }
  CU_TRY(ctx, cudaMemcpyAsync(out, dout.p, 32 * n_items, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

extern "C" int cdx_hash_cells_dev(cdx_ctx* ctx, const void* d_data, size_t n_cells, size_t cell_size, void* d_out, void* stream) {
  if (!ctx || !d_data || !d_out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (cell_size == 0 || cell_size % 4 || cell_size > (1u << 30)) return fail(ctx, CDX_ERR_SIZE, "cell size %zu must be a non-zero multiple of 4", cell_size);
  if ((uintptr_t)d_data % 16 || (uintptr_t)d_out % 16) return fail(ctx, CDX_ERR_ARG, "buffers must be 16-byte aligned");
  if (n_cells == 0) return CDX_OK;
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  return launch_hash_cells(ctx, d_data, n_cells, cell_size, (uint8_t*)d_out, st);
}

extern "C" int cdx_compress_batch_host(cdx_ctx* ctx, const uint8_t* x, const uint8_t* y, const uint32_t* keys, size_t n, uint8_t* out) {
  if (!ctx || !x || !y || !keys || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  for (size_t i = 0; i < n; ++i)
    if (keys[i] > 3) return fail(ctx, CDX_ERR_ARG, "key %u at %zu is not in 0..3", keys[i], i);
  if (n == 0) return CDX_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf dx, dy, dk, dout;
  CU_TRY(ctx, dx.alloc(32 * n, ctx->stream));
  CU_TRY(ctx, dy.alloc(32 * n, ctx->stream));
  CU_TRY(ctx, dk.alloc(4 * n, ctx->stream));
  CU_TRY(ctx, dout.alloc(32 * n, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(dx.p, x, 32 * n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(dy.p, y, 32 * n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(dk.p, keys, 4 * n, cudaMemcpyHostToDevice, ctx->stream));
  LAUNCH(ctx, k_compress_batch, n, ctx->stream, dx.u8(), dy.u8(), (const uint32_t*)dk.p, n, dout.u8());
  CU_TRY(ctx, cudaMemcpyAsync(out, dout.p, 32 * n, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

// ---- Merkle trees -------------------------------------------------------------------------------------------

extern "C" size_t cdx_merkle_total_nodes(size_t n, int bottom_layer) {
  if (n == 0) return 0;
  size_t total = 0;
  bool bottom = bottom_layer != 0;
  for (;;) {
    total += n;
    if (!bottom && n == 1) return total;
    n = (n + 1) / 2;
    bottom = false;
  }
}

extern "C" int cdx_merkle_num_layers(size_t n, int bottom_layer) {
  if (n == 0) return 0;
  int layers = 1;
  bool bottom = bottom_layer != 0;
  for (;;) {
    if (!bottom && n == 1) return layers;
    n = (n + 1) / 2;
    bottom = false;
    ++layers;
  }
}

// builds every level above d_layers[0..n) in place (layers concatenated); level kernels run back to back on st
static int merkle_layers_on_device(cdx_ctx* ctx, uint8_t* d_layers, size_t n, bool bottom, cudaStream_t st) {
  uint8_t* cur = d_layers;
  for (;;) {
    if (!bottom && n == 1) return CDX_OK;
    uint8_t* next = cur + 32 * n;
    LAUNCH(ctx, k_merkle_level, (n + 1) / 2, st, cur, n, next, bottom ? 1u : 0u, 0);
    cur = next;
    n = (n + 1) / 2;
    bottom = false;
  }
}

extern "C" int cdx_merkle_layers_host(cdx_ctx* ctx, const uint8_t* leaves, size_t n, int bottom_layer, uint8_t* layers_out) {
  if (!ctx || !leaves || !layers_out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (n == 0) return fail(ctx, CDX_ERR_ARG, "merkle tree of empty input");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t total = cdx_merkle_total_nodes(n, bottom_layer);
  DevBuf d;
  CU_TRY(ctx, d.alloc(32 * total, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(d.p, leaves, 32 * n, cudaMemcpyHostToDevice, ctx->stream));
  LAUNCH(ctx, k_canonical_felts, n, ctx->stream, d.u8(), n);       // layer 0 is returned too: leaves >= r come back mod r
  int rc = merkle_layers_on_device(ctx, d.u8(), n, bottom_layer != 0, ctx->stream);
  if (rc) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(layers_out, d.p, 32 * total, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

extern "C" int cdx_merkle_root_host(cdx_ctx* ctx, const uint8_t* leaves, size_t n, uint8_t root_out[32]) {
  if (!ctx || !leaves || !root_out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (n == 0) return fail(ctx, CDX_ERR_ARG, "merkle tree of empty input");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t total = cdx_merkle_total_nodes(n, 1);
  DevBuf d;
  CU_TRY(ctx, d.alloc(32 * total, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(d.p, leaves, 32 * n, cudaMemcpyHostToDevice, ctx->stream));
  int rc = merkle_layers_on_device(ctx, d.u8(), n, true, ctx->stream);
  if (rc) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(root_out, d.u8() + 32 * (total - 1), 32, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

// ---- slot commitment ----------------------------------------------------------------------------------------

static bool is_pow2(uint64_t x) { return x && !(x & (x - 1)); }
static uint32_t log2_u64(uint64_t x) {
  uint32_t k = 0;
  while ((1ull << k) < x) ++k;
  return k;
}

extern "C" void cdx_slot_free(cdx_slot* s) {
  if (!s) return;
  if (s->ctx) cudaSetDevice(s->ctx->device);
  if (s->d_forest) dev_free(s->d_forest, s->stream);   // ordered after everything queued on the slot's stream
  if (s->d_low) dev_free(s->d_low, s->stream);
  if (s->d_top) dev_free(s->d_top, s->stream);
  delete s;
}

static int check_shape(cdx_ctx* ctx, size_t n_bytes, size_t cell_size, size_t block_size) {
  char msg[128];
  const int rc = slot_shape_status(n_bytes, cell_size, block_size, msg, sizeof msg);
  return rc ? fail(ctx, rc, "%s", msg) : CDX_OK;
}

// allocate a slot handle and lay out its layers; on success the caller fills forest[0] and calls build_trees
// n_local_blocks == 0 is an EMPTY SHARD (a rank that got no chunk of a small slot): it holds nothing below top_level, takes part
// in the exchange with zero nodes and still gets the replicated top tree; only the sharded entry points create one.
// compact: a whole slot that keeps only the block hashes of its forest (a compact image being imported).
static int slot_alloc(cdx_ctx* ctx, uint64_t n_local_blocks, size_t cell_size, size_t block_size, uint64_t first_block,
                      uint64_t n_total_blocks, int top_level, cudaStream_t st, cdx_slot** out, bool allow_empty = false, bool compact = false) {
  const uint64_t cpb = block_size / cell_size;
  if (n_total_blocks == 0 || (n_local_blocks == 0 && !allow_empty) || first_block + n_local_blocks > n_total_blocks)
    return fail(ctx, CDX_ERR_RANGE, "block range [%llu,+%llu) outside slot of %llu blocks", (unsigned long long)first_block,
                (unsigned long long)n_local_blocks, (unsigned long long)n_total_blocks);
  cdx_slot* s = new (std::nothrow) cdx_slot();
  if (!s) return fail(ctx, CDX_ERR_ALLOC, "host allocation failed");
  s->ctx = ctx;
  s->stream = st;
  s->cell_size = cell_size;
  s->block_size = block_size;
  s->n_local_blocks = n_local_blocks;
  s->n_local_cells = n_local_blocks * cpb;
  s->first_block = first_block;
  s->n_total_blocks = n_total_blocks;
  s->cpb_log2 = log2_u64(cpb);
  s->block_depth = cpb == 1 ? 1 : s->cpb_log2;
  // global widths of the slot tree (merkle/bn254.nim:29-60): n, ceil(n/2), ..., 1; a single block still gets
  // one key-3 compression
  {
    uint64_t w = n_total_blocks;
    bool bottom = true;
    for (;;) {
      s->width.push_back(w);
      if (!bottom && w == 1) break;
      w = (w + 1) / 2;
      bottom = false;
    }
    s->slot_depth = (uint32_t)s->width.size() - 1;
  }
  if (top_level < 0 || (uint32_t)top_level > s->slot_depth || (n_total_blocks == 1 && top_level != 0)) {
    const uint32_t depth = s->slot_depth;
    delete s;
    return fail(ctx, CDX_ERR_RANGE, "top_level %d outside 0..%u", top_level, depth);
  }
  s->top_level = (uint32_t)top_level;
  const uint64_t align = 1ull << top_level;
  if (first_block % align || (n_local_blocks % align && first_block + n_local_blocks != n_total_blocks)) {
    delete s;
    return fail(ctx, CDX_ERR_SIZE, "block range is not aligned to 2^top_level");
  }
  // forest: levels 0..block_depth
  size_t forest_nodes = 0;
  std::vector<size_t> f_off;
  for (uint32_t l = 0; l <= s->block_depth; ++l) {
    f_off.push_back(compact ? 0 : forest_nodes);
    if (!compact || l == s->block_depth) forest_nodes += cpb == 1 ? s->n_local_cells : (s->n_local_cells >> l);
  }
  // low: slot levels 1..top_level over the local range
  size_t low_nodes = 0;
  std::vector<size_t> l_off;
  s->low_first.assign(s->top_level + 1, 0);
  s->low_count.assign(s->top_level + 1, 0);
  s->low_first[0] = first_block;
  s->low_count[0] = n_local_blocks;
  l_off.push_back(0);
  for (uint32_t l = 1; l <= s->top_level; ++l) {
    s->low_first[l] = first_block >> l;
    s->low_count[l] = (s->low_count[l - 1] + 1) / 2;
    l_off.push_back(low_nodes);
    low_nodes += s->low_count[l];
  }
  cudaError_t e = forest_nodes ? dev_alloc((void**)&s->d_forest, 32 * forest_nodes, st) : cudaSuccess;
  if (e == cudaSuccess && low_nodes) e = dev_alloc((void**)&s->d_low, 32 * low_nodes, st);
  if (e != cudaSuccess) {
    cdx_slot_free(s);
    return fail(ctx, CDX_ERR_ALLOC, "cudaMalloc of %zu tree nodes failed: %s", forest_nodes + low_nodes, cudaGetErrorString(e));
  }
  for (uint32_t l = 0; l <= s->block_depth; ++l) s->forest.push_back(compact && l < s->block_depth ? nullptr : s->d_forest + 32 * f_off[l]);
  s->compact = compact;
  s->low.push_back(s->forest[s->block_depth]);
  for (uint32_t l = 1; l <= s->top_level; ++l) s->low.push_back(s->d_low + 32 * l_off[l]);
  *out = s;
  return CDX_OK;
}

// The block trees over n_cells cell hashes of whole blocks in forest[0]: levels 1..block_depth into forest[1..block_depth],
// one launch per level (one launch for one-cell blocks, whose single level is one key-3 compression per cell).
static int launch_block_trees(cdx_ctx* ctx, uint8_t* const* forest, size_t n_cells, bool singles, uint32_t block_depth, cudaStream_t st) {
  if (singles) {
    LAUNCH(ctx, k_merkle_level, n_cells, st, forest[0], n_cells, forest[1], 1u, 1);
  } else {
    for (uint32_t l = 0; l < block_depth; ++l) {
      const size_t n = n_cells >> l;
      LAUNCH(ctx, k_merkle_level, n / 2, st, forest[l], n, forest[l + 1], l == 0 ? 1u : 0u, 0);
    }
  }
  return CDX_OK;
}

// block forest + local slot levels, assuming forest[0] (cell hashes) is already being produced on s->stream
static int build_local_trees(cdx_slot* s) {
  cdx_ctx* ctx = s->ctx;
  const bool singles = (s->block_size / s->cell_size) == 1;
  if (s->n_local_cells == 0) return CDX_OK;                                  // empty shard
  int rc = launch_block_trees(ctx, s->forest.data(), (size_t)s->n_local_cells, singles, s->block_depth, s->stream);
  if (rc) return rc;
  for (uint32_t l = 0; l < s->top_level; ++l) {
    const size_t n = s->low_count[l];
    LAUNCH(ctx, k_merkle_level, (n + 1) / 2, s->stream, s->low[l], n, s->low[l + 1], l == 0 ? 1u : 0u, 0);
  }
  return CDX_OK;
}

// upper (replicated) levels from the complete level-top_level layer
static int build_top(cdx_slot* s, const uint8_t* d_level_nodes, bool alias) {
  cdx_ctx* ctx = s->ctx;
  const uint32_t T = s->top_level;
  size_t nodes = 0;
  std::vector<size_t> off;
  for (uint32_t l = T; l <= s->slot_depth; ++l) {
    off.push_back(nodes);
    if (!(alias && l == T)) nodes += s->width[l];
  }
  if (s->d_top) {
    dev_free(s->d_top, s->stream);
    s->d_top = nullptr;
  }
  if (nodes) CU_TRY(ctx, dev_alloc((void**)&s->d_top, 32 * nodes, s->stream));
  s->top.assign(s->slot_depth + 1, nullptr);
  for (uint32_t l = T; l <= s->slot_depth; ++l) s->top[l] = s->d_top + 32 * off[l - T];
  if (alias) {
    s->top[T] = const_cast<uint8_t*>(d_level_nodes);
  } else {
    CU_TRY(ctx, cudaMemcpyAsync(s->top[T], d_level_nodes, 32 * s->width[T], cudaMemcpyDeviceToDevice, s->stream));
  }
  s->top0_alias = alias;
  for (uint32_t l = T; l < s->slot_depth; ++l) {
    const size_t n = s->width[l];
    LAUNCH(ctx, k_merkle_level, (n + 1) / 2, s->stream, s->top[l], n, s->top[l + 1], l == 0 ? 1u : 0u, 0);
  }
  s->has_top = true;
  return CDX_OK;
}

extern "C" int cdx_slot_commit_range_dev(cdx_ctx* ctx, const void* d_data, size_t n_local_bytes, size_t cell_size, size_t block_size,
                                         uint64_t first_block, uint64_t n_total_blocks, int top_level, void* stream, cdx_slot** out) {
  if (!ctx || !d_data || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  int rc = check_shape(ctx, n_local_bytes, cell_size, block_size);
  if (rc) return rc;
  if ((uintptr_t)d_data % 16) return fail(ctx, CDX_ERR_ARG, "slot data must be 16-byte aligned");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  cdx_slot* s = nullptr;
  rc = slot_alloc(ctx, n_local_bytes / block_size, cell_size, block_size, first_block, n_total_blocks, top_level, st, &s);
  if (rc) return rc;
  auto body = [&]() -> int {
    int r = launch_hash_cells(ctx, d_data, (size_t)s->n_local_cells, cell_size, s->forest[0], st);
    if (r) return r;
    return build_local_trees(s);
  };
  rc = body();
  if (rc) {
    cdx_slot_free(s);
    return rc;
  }
  *out = s;
  return CDX_OK;
}

extern "C" int cdx_slot_commit_dev(cdx_ctx* ctx, const void* d_data, size_t n_bytes, size_t cell_size, size_t block_size, void* stream, cdx_slot** out) {
  if (!ctx || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (block_size == 0) return fail(ctx, CDX_ERR_SIZE, "block size is zero");
  cdx_slot* s = nullptr;
  int rc = cdx_slot_commit_range_dev(ctx, d_data, n_bytes, cell_size, block_size, 0, n_bytes / block_size, 0, stream, &s);
  if (rc) return rc;
  rc = build_top(s, s->low[0], true);
  if (rc) {
    cdx_slot_free(s);
    return rc;
  }
  *out = s;
  return CDX_OK;
}

static int ensure_stage(cdx_ctx* ctx, size_t bytes, int count = 2) {
  if (ctx->stage_bytes >= bytes && ctx->stage_count >= count) return CDX_OK;
  const size_t want_bytes = bytes > ctx->stage_bytes ? bytes : ctx->stage_bytes;
  const int want_count = count > ctx->stage_count ? count : ctx->stage_count;
  CU_TRY(ctx, cudaDeviceSynchronize());                       // earlier calls may still be reading the old tiles
  release_stage(ctx);
  for (int i = 0; i < want_count; ++i) CU_TRY(ctx, dev_alloc(&ctx->d_stage[i], want_bytes, ctx->stream, false));
  ctx->stage_bytes = want_bytes;
  ctx->stage_count = want_count;
  return CDX_OK;
}

// ---- cell-hash pipelines: slot bytes that are not resident in HBM -------------------------------------------------
// Every source that is not in HBM (pinned or pageable host memory, a file, generated bytes) reaches the cell sponge
// through run_tiles.  The slot is cut into tiles of whole blocks.  Tile t is produced into staging buffer t % n_bufs and
// hashed on compute stream t & 1: two compute streams let the sponge kernels of consecutive tiles overlap at the seams
// (the tail of one fills up with the head of the next).  Each buffer is reused strictly in order: the producer of tile t
// waits for the sponge of tile t - n_bufs, and the sponge of tile t waits for its producer.  The pipelines differ only
// in their tile sizes, their number of buffers and their producer.  They return with ctx->stream ordered after all of
// their work (no host sync); the caller continues on ctx->stream.
typedef std::function<void(uint8_t* dst, uint64_t offset, size_t len)> ChunkFill;

static void drain_streams(cdx_ctx* ctx) {
  cudaStreamSynchronize(ctx->copy_stream);
  cudaStreamSynchronize(ctx->copy_stream2);
  cudaStreamSynchronize(ctx->stream2);
  cudaStreamSynchronize(ctx->stream);
}

// An open slot data file as a ChunkFill.  A read error is not an end of file: EINTR is retried, anything else is
// recorded (the fill runs on worker threads) and fails the commit; only a true EOF zero-fills, like the reference's
// ignored short reads (slot.nim:64-65).
struct FileSource {
  int fd = -1;
  uint64_t base = 0;
  std::atomic<int> io_errno{0};
  ChunkFill fill;
  ~FileSource() {
    if (fd >= 0) close(fd);
  }
  bool open_path(const char* path, uint64_t base_offset) {
    fd = open(path, O_RDONLY);
    base = base_offset;
    fill = [this](uint8_t* dst, uint64_t off, size_t len) {
      size_t pos = 0;
      while (pos < len) {
        const ssize_t got = pread(fd, dst + pos, len - pos, (off_t)(base + off + pos));
        if (got < 0) {
          if (errno == EINTR) continue;
          int expected = 0;
          io_errno.compare_exchange_strong(expected, errno);
          break;
        }
        if (got == 0) break;
        pos += (size_t)got;
      }
      if (pos < len) memset(dst + pos, 0, len - pos);
    };
    return fd >= 0;
  }
};

// tile sizes in blocks: `head`, then `tile` until n_blocks are covered; the last tile is clipped to what remains
static std::vector<size_t> tile_schedule(size_t n_blocks, const std::vector<size_t>& head, size_t tile) {
  std::vector<size_t> tiles;
  for (size_t done = 0; done < n_blocks; done += tiles.back()) {
    const size_t want = tiles.size() < head.size() ? head[tiles.size()] : tile;
    tiles.push_back(n_blocks - done < want ? n_blocks - done : want);
  }
  return tiles;
}

// queues the bytes of blocks [first, first + nb), which make up tile t, into the staging buffer dst on stream st
typedef std::function<int(int t, size_t first, size_t nb, uint8_t* dst, cudaStream_t st)> TileProducer;

// Tiles with an even index are produced on `even`, those with an odd index on `odd`; a null stream produces the tile on
// its compute stream.  Only these streams and ctx->stream2 are ordered after the caller's earlier work on ctx->stream: a
// copy stream held up for nothing would also hold up upload_table, whose next call waits on the host for the last one.
// `consume` (may be null) queues more work on a tile, on its compute stream after its sponge, before the buffer is reused.
static int run_tiles(cdx_ctx* ctx, const std::vector<size_t>& tiles, int n_bufs, cudaStream_t even, cudaStream_t odd, size_t cell_size,
                     size_t block_size, const TileProducer& produce, uint8_t* d_hashes, const TileProducer* consume = nullptr) {
  CU_TRY(ctx, cudaEventRecord(ctx->ev_join, ctx->stream));              // d_hashes was allocated on ctx->stream, and
  CU_TRY(ctx, cudaStreamWaitEvent(ctx->stream2, ctx->ev_join, 0));      // earlier work on it may still read the buffers
  if (even) CU_TRY(ctx, cudaStreamWaitEvent(even, ctx->ev_join, 0));
  if (odd && odd != even) CU_TRY(ctx, cudaStreamWaitEvent(odd, ctx->ev_join, 0));
  const size_t cpb = block_size / cell_size;
  size_t first = 0;
  for (int t = 0; t < (int)tiles.size(); ++t) {
    const int b = t % n_bufs;
    const size_t nb = tiles[t];
    cudaStream_t cs = (t & 1) ? ctx->stream2 : ctx->stream;
    cudaStream_t ps = (t & 1) ? odd : even;
    if (!ps) ps = cs;
    if (t >= n_bufs) CU_TRY(ctx, cudaStreamWaitEvent(ps, ctx->ev_consumed[b], 0));
    int rc = produce(t, first, nb, (uint8_t*)ctx->d_stage[b], ps);
    if (rc) return rc;
    if (ps != cs) {
      CU_TRY(ctx, cudaEventRecord(ctx->ev_copied[b], ps));
      CU_TRY(ctx, cudaStreamWaitEvent(cs, ctx->ev_copied[b], 0));
    }
    rc = launch_hash_cells(ctx, ctx->d_stage[b], nb * cpb, cell_size, d_hashes + 32 * first * cpb, cs);
    if (rc) return rc;
    if (consume) {
      rc = (*consume)(t, first, nb, (uint8_t*)ctx->d_stage[b], cs);
      if (rc) return rc;
    }
    CU_TRY(ctx, cudaEventRecord(ctx->ev_consumed[b], cs));
    first += nb;
  }
  CU_TRY(ctx, cudaEventRecord(ctx->ev_join, ctx->stream2));             // the caller's trees run on ctx->stream after both
  CU_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));       // compute streams
  return CDX_OK;
}

// Pinned (or otherwise DMA-able) host memory: one copy per tile, on copy stream t & 1.  NS = 3 buffers and two copy
// streams keep TWO copies in flight ahead of the sponge, which rides out a host whose PCIe/memory path is shared by eight
// GPUs streaming at once (DESIGN.md section 7).
static int hash_cells_pinned(cdx_ctx* ctx, const uint8_t* data, size_t n_bytes, size_t cell_size, size_t block_size, uint8_t* d_hashes) {
  const size_t n_blocks = n_bytes / block_size;
  // Tile = 256 MiB: 131 072 cells of 2 KiB, about one full wave of the cell-sponge kernel on 148 SMs (the resident
  // CTAs per SM are set by CDX_TMA_MIN_CTAS in kernels.cuh); smaller tiles leave SMs idle, larger ones only add exposed
  // first-copy latency.  Slots below 1 GiB are cut in four so that the copy still overlaps.
  size_t tile_bytes_target = ctx->tile_mib << 20;
  if (n_bytes < ((size_t)1 << 30)) tile_bytes_target = n_bytes / 4 > ((size_t)16 << 20) ? n_bytes / 4 : ((size_t)16 << 20);
  size_t tile_blocks = tile_bytes_target / block_size;
  if (tile_blocks == 0) tile_blocks = 1;
  if (tile_blocks > n_blocks) tile_blocks = n_blocks;
  const int NS = ctx->stage_tiles;
  int rc = ensure_stage(ctx, tile_blocks * block_size, NS);
  if (rc) return rc;
  // Start of the pipeline.  The copy of tile 0 is the only one nothing overlaps, so it is short; after that the copy of
  // tile t+1 has to hide behind the sponge of tile t.  Two starts:
  //   mode 0  1/8 tile, then 7/8 (realigns with the tile grid);
  //   mode 1  gradual: tiles grow by a quarter per step from 1/4 tile.
  // Measured (profiles/r2_e2e_sweep_ramp_n1.txt, r2_e2e_sweep_ramp_n8.txt): the gradual start gains 0.5 % end to end when this
  // GPU has the host's PCIe/memory path to itself (H2D 55 GB/s) and LOSES 0.7 % when eight GPUs share it (23-35 GB/s per
  // GPU).  So the default (mode 2) decides per call from the H2D rate this context measured on its previous pinned
  // commit (two events around one full-size tile copy, read back here without waiting): gradual above 48 GB/s, else
  // mode 0; the first commit of a context uses mode 0.  CODEX_COMMIT_RAMP=0/1 pins the choice.
  if (ctx->rate_bytes) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev_rate[0], ctx->ev_rate[1]) == cudaSuccess && ms > 0.f) {
      ctx->h2d_gbs = (double)ctx->rate_bytes / (ms * 1e6);
      ctx->rate_bytes = 0;
    } else {
      cudaGetLastError();                                               // not finished yet (cannot happen after a synchronised commit)
    }
  }
  const bool gradual = ctx->ramp_mode == 1 || (ctx->ramp_mode == 2 && ctx->h2d_gbs > 48.0);
  std::vector<size_t> head;
  if (n_blocks > tile_blocks && tile_blocks >= 8) {
    if (gradual) {
      for (size_t cur = tile_blocks / 4; cur < tile_blocks; cur += cur / 4 ? cur / 4 : 1) head.push_back(cur);
    } else {
      head = {tile_blocks / 8, tile_blocks - tile_blocks / 8};
    }
  }
  bool rate_armed = false;
  auto copy = [&](int t, size_t first, size_t nb, uint8_t* dst, cudaStream_t cp) -> int {
    const bool measure = !rate_armed && nb == tile_blocks && t >= NS;    // a full tile in steady state (its buffer wait is already behind it)
    if (measure) CU_TRY(ctx, cudaEventRecord(ctx->ev_rate[0], cp));
    CU_TRY(ctx, cudaMemcpyAsync(dst, data + first * block_size, nb * block_size, cudaMemcpyHostToDevice, cp));
    if (measure) {
      CU_TRY(ctx, cudaEventRecord(ctx->ev_rate[1], cp));
      ctx->rate_bytes = nb * block_size;
      rate_armed = true;
    }
    return CDX_OK;
  };
  return run_tiles(ctx, tile_schedule(n_blocks, head, tile_blocks), NS, ctx->copy_stream, ctx->copy_stream2, cell_size, block_size, copy,
                   d_hashes);
}

// len bytes of a source at offset off into dst through `fill`, split evenly over host threads (8 on a host with 16 or more
// hardware threads, 4 with 8 or more, else 2): one thread copying pageable memory into pinned memory does not keep up
// with the cell sponge.
static void fill_chunk_parallel(const ChunkFill& fill, uint8_t* dst, uint64_t off, size_t len) {
  const unsigned hw = std::thread::hardware_concurrency();
  const unsigned n_thr = hw >= 16 ? 8 : (hw >= 8 ? 4 : 2);
  std::vector<std::thread> thr;
  for (unsigned t = 0; t < n_thr; ++t) {
    const size_t a = len * t / n_thr, b = len * (t + 1) / n_thr;
    if (b > a) thr.emplace_back([&fill, dst, off, a, b]() { fill(dst + a, off + a, b - a); });
  }
  for (auto& t : thr) t.join();
}

// Slot bytes that are not directly DMA-able (a file, or pageable host memory -- what a Nim seq[byte] is).  Host threads
// fill one of two pinned chunks through `fill(dst, offset, len)` while the copy stream moves the other one into the
// device tile; a tile is four chunks, copied on the one copy stream into two device buffers.
static int hash_cells_staged(cdx_ctx* ctx, size_t n_bytes, size_t cell_size, size_t block_size, const ChunkFill& fill, uint8_t* d_hashes,
                             const TileProducer* consume = nullptr) {
  const size_t n_blocks = n_bytes / block_size;
  const size_t chunk_bytes_target = (ctx->tile_mib << 20) / 4;              // pinned chunk
  size_t chunk_blocks = chunk_bytes_target / block_size ? chunk_bytes_target / block_size : 1;
  size_t tile_blocks = 4 * chunk_blocks;                                    // device tile = 4 chunks = 256 MiB (one sponge wave)
  if (tile_blocks > n_blocks) tile_blocks = n_blocks;
  if (chunk_blocks > tile_blocks) chunk_blocks = tile_blocks;
  const size_t chunk_bytes = chunk_blocks * block_size, tile_bytes = tile_blocks * block_size;
  if (ctx->pinned_bytes < chunk_bytes) {
    for (int i = 0; i < 2; ++i) {
      if (ctx->h_pinned[i]) cudaFreeHost(ctx->h_pinned[i]);
      ctx->h_pinned[i] = nullptr;
    }
    ctx->pinned_bytes = 0;
    for (int i = 0; i < 2; ++i)
      if (cudaHostAlloc(&ctx->h_pinned[i], chunk_bytes, cudaHostAllocDefault) != cudaSuccess)
        return fail(ctx, CDX_ERR_ALLOC, "cudaHostAlloc of %zu bytes failed", chunk_bytes);
    ctx->pinned_bytes = chunk_bytes;
  }
  int rc = ensure_stage(ctx, tile_bytes);
  if (rc) return rc;
  // tile 0 is one chunk, tile 1 the other three: the sponge starts after one chunk has been filled and copied, not four
  std::vector<size_t> head;
  if (n_blocks > tile_blocks && tile_blocks > chunk_blocks) head = {chunk_blocks, tile_blocks - chunk_blocks};
  size_t chunk_no = 0;
  auto copy = [&](int, size_t first, size_t nb, uint8_t* dst, cudaStream_t cp) -> int {
    for (size_t cb = 0; cb < nb; cb += chunk_blocks, ++chunk_no) {
      const int pb = (int)(chunk_no & 1);
      const size_t cnb = nb - cb < chunk_blocks ? nb - cb : chunk_blocks;
      if (chunk_no >= 2) CU_TRY(ctx, cudaEventSynchronize(ctx->ev_h2d[pb]));                  // pinned chunk pb drained
      fill_chunk_parallel(fill, (uint8_t*)ctx->h_pinned[pb], (uint64_t)(first + cb) * block_size, cnb * block_size);
      CU_TRY(ctx, cudaMemcpyAsync(dst + cb * block_size, ctx->h_pinned[pb], cnb * block_size, cudaMemcpyHostToDevice, cp));
      CU_TRY(ctx, cudaEventRecord(ctx->ev_h2d[pb], cp));
    }
    return CDX_OK;
  };
  rc = run_tiles(ctx, tile_schedule(n_blocks, head, tile_blocks), 2, ctx->copy_stream, ctx->copy_stream, cell_size, block_size, copy, d_hashes,
                 consume);
  if (rc) return rc;
  // the pinned chunks are reused by the next call: their last copies must have left the host
  CU_TRY(ctx, cudaEventSynchronize(ctx->ev_h2d[0]));
  if (chunk_no >= 2) CU_TRY(ctx, cudaEventSynchronize(ctx->ev_h2d[1]));
  return CDX_OK;
}

// Host memory of either kind.  Pageable memory (an ordinary malloc / Nim seq) is copied by the driver through one staging
// thread at ~11 GB/s, below the sponge rate; several host threads copying into our own pinned chunks keep up with it.
static int hash_cells_host(cdx_ctx* ctx, const uint8_t* data, size_t n_bytes, size_t cell_size, size_t block_size, uint8_t* d_hashes) {
  if (n_bytes >= ((size_t)256 << 20) && !ctx->no_bounce) {
    cudaPointerAttributes attr;
    const cudaError_t e = cudaPointerGetAttributes(&attr, data);
    if (e != cudaSuccess) cudaGetLastError();
    if (e != cudaSuccess || attr.type == cudaMemoryTypeUnregistered) {
      ChunkFill fill = [data](uint8_t* dst, uint64_t off, size_t len) { memcpy(dst, data + off, len); };
      return hash_cells_staged(ctx, n_bytes, cell_size, block_size, fill, d_hashes);
    }
  }
  return hash_cells_pinned(ctx, data, n_bytes, cell_size, block_size, d_hashes);
}

// Generated slot bytes (the reference's fake data or the benchmark's counter-based bytes): the generator kernel writes a
// device tile on the tile's compute stream, two tiles in flight.  Nothing crosses PCIe and no slot-sized buffer exists,
// so a 100 GiB slot costs 512 MiB of staging.  first_byte is the offset of this range inside its slot.
static int launch_fake_cells(cdx_ctx* ctx, uint64_t seed, uint64_t first_cell, size_t n_cells, size_t cell_size, void* d_out, cudaStream_t st);
static int launch_fill_synthetic(cdx_ctx* ctx, uint64_t seed, uint64_t first_word, size_t n_bytes, void* d_out, cudaStream_t st);
static int fill_synthetic_range(cdx_ctx* ctx, uint64_t seed, uint64_t first_byte, size_t n_bytes, void* d_out, cudaStream_t st);
static int generate_bytes(cdx_ctx* ctx, uint32_t kind, uint64_t seed, uint64_t first_byte, size_t n_bytes, size_t cell_size, void* d_out, cudaStream_t st) {
  if (kind == CDX_SRC_FAKE) return launch_fake_cells(ctx, seed, first_byte / cell_size, n_bytes / cell_size, cell_size, d_out, st);
  return fill_synthetic_range(ctx, seed, first_byte, n_bytes, d_out, st);
}
static int hash_cells_generated(cdx_ctx* ctx, uint32_t kind, uint64_t seed, uint64_t first_byte, size_t n_bytes, size_t cell_size, size_t block_size,
                                uint8_t* d_hashes) {
  const size_t n_blocks = n_bytes / block_size;
  size_t tile_blocks = (ctx->tile_mib << 20) / block_size;
  if (tile_blocks == 0) tile_blocks = 1;
  if (tile_blocks > n_blocks) tile_blocks = n_blocks;
  int rc = ensure_stage(ctx, tile_blocks * block_size);
  if (rc) return rc;
  auto generate = [&](int, size_t first, size_t nb, uint8_t* dst, cudaStream_t st) {
    return generate_bytes(ctx, kind, seed, first_byte + first * block_size, nb * block_size, cell_size, dst, st);
  };
  return run_tiles(ctx, tile_schedule(n_blocks, {}, tile_blocks), 2, nullptr, nullptr, cell_size, block_size, generate, d_hashes);
}

// where the bytes of a slot (or of a block range of one) come from
struct SlotSource {
  uint32_t kind = CDX_SRC_HOST;
  uint64_t seed = 0;
  const uint8_t* host = nullptr;        // CDX_SRC_HOST: first byte of the RANGE
  const ChunkFill* fill = nullptr;      // CDX_SRC_FILE: reads range-relative offsets
  uint64_t first_byte = 0;              // generated kinds: offset of the range inside its slot
};

static int hash_cells_source(cdx_ctx* ctx, const SlotSource& src, size_t n_bytes, size_t cell_size, size_t block_size, uint8_t* d_hashes) {
  switch (src.kind) {
    case CDX_SRC_HOST: return hash_cells_host(ctx, src.host, n_bytes, cell_size, block_size, d_hashes);
    case CDX_SRC_FILE: return hash_cells_staged(ctx, n_bytes, cell_size, block_size, *src.fill, d_hashes);
    case CDX_SRC_FAKE:
    case CDX_SRC_SYNTHETIC: return hash_cells_generated(ctx, src.kind, src.seed, src.first_byte, n_bytes, cell_size, block_size, d_hashes);
    default: return fail(ctx, CDX_ERR_ARG, "unknown slot source kind %u", src.kind);
  }
}

// A slot (whole_slot) or a block range of one, from any non-resident source: cell hashes through the matching pipeline,
// then block trees and the local slot levels (and the top tree for a whole slot) on ctx->stream.  With `sync` it returns
// synchronised (the public single-slot entry points); without, the work is queued and the source bytes must stay valid
// until the caller synchronises (the dataset commit queues all of a rank's slots and waits once).
// n_bytes == 0 is an empty shard (sharded entry points only).
static int commit_from_source(cdx_ctx* ctx, const SlotSource& src, size_t n_bytes, size_t cell_size, size_t block_size, uint64_t first_block,
                              uint64_t n_total_blocks, int top_level, bool whole_slot, bool sync, cdx_slot** out) {
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n_blocks = n_bytes / block_size;
  if (whole_slot) n_total_blocks = n_blocks;
  cdx_slot* s = nullptr;
  int rc = slot_alloc(ctx, n_blocks, cell_size, block_size, first_block, n_total_blocks, top_level, ctx->stream, &s, !whole_slot);
  if (rc) return rc;
  auto body = [&]() -> int {
    if (n_blocks) {
      int r = hash_cells_source(ctx, src, n_bytes, cell_size, block_size, s->forest[0]);
      if (r) return r;
      r = build_local_trees(s);
      if (r) return r;
    }
    if (whole_slot) {
      int r = build_top(s, s->low[0], true);
      if (r) return r;
    }
    if (sync) CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return CDX_OK;
  };
  rc = body();
  if (rc) {
    drain_streams(ctx);
    cdx_slot_free(s);
    return rc;
  }
  *out = s;
  return CDX_OK;
}

static int commit_host_range(cdx_ctx* ctx, const uint8_t* data, size_t n_bytes, size_t cell_size, size_t block_size, uint64_t first_block,
                             uint64_t n_total_blocks, int top_level, bool whole_slot, cdx_slot** out) {
  if (!ctx || !data || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  int rc = check_shape(ctx, n_bytes, cell_size, block_size);
  if (rc) return rc;
  SlotSource src;
  src.kind = CDX_SRC_HOST;
  src.host = data;
  return commit_from_source(ctx, src, n_bytes, cell_size, block_size, first_block, n_total_blocks, top_level, whole_slot, true, out);
}

extern "C" int cdx_slot_commit_host(cdx_ctx* ctx, const uint8_t* data, size_t n_bytes, size_t cell_size, size_t block_size, cdx_slot** out) {
  return commit_host_range(ctx, data, n_bytes, cell_size, block_size, 0, 0, 0, true, out);
}

extern "C" int cdx_slot_commit_range_host(cdx_ctx* ctx, const uint8_t* data, size_t n_local_bytes, size_t cell_size, size_t block_size,
                                          uint64_t first_block, uint64_t n_total_blocks, int top_level, cdx_slot** out) {
  return commit_host_range(ctx, data, n_local_bytes, cell_size, block_size, first_block, n_total_blocks, top_level, false, out);
}

extern "C" int cdx_slot_commit_file(cdx_ctx* ctx, const char* path, uint64_t offset, size_t n_bytes, size_t cell_size, size_t block_size, cdx_slot** out) {
  if (!ctx || !path || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  int rc = check_shape(ctx, n_bytes, cell_size, block_size);
  if (rc) return rc;
  FileSource file;
  if (!file.open_path(path, offset)) return fail(ctx, CDX_ERR_ARG, "cannot open slot data file `%s`", path);
  SlotSource src;
  src.kind = CDX_SRC_FILE;
  src.fill = &file.fill;
  rc = commit_from_source(ctx, src, n_bytes, cell_size, block_size, 0, 0, 0, true, true, out);
  if (rc == CDX_OK && file.io_errno.load() != 0) {
    cdx_slot_free(*out);
    *out = nullptr;
    return fail(ctx, CDX_ERR_ARG, "reading slot data file `%s` failed: %s", path, strerror(file.io_errno.load()));
  }
  return rc;
}

extern "C" int cdx_slot_commit_fake(cdx_ctx* ctx, uint64_t seed, size_t n_cells, size_t cell_size, size_t block_size, cdx_slot** out) {
  if (!ctx || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  if (cell_size == 0 || n_cells == 0 || n_cells > ((size_t)1 << 40) / cell_size) return fail(ctx, CDX_ERR_SIZE, "bad fake slot size");
  int rc = check_shape(ctx, n_cells * cell_size, cell_size, block_size);
  if (rc) return rc;
  SlotSource src;
  src.kind = CDX_SRC_FAKE;
  src.seed = seed;
  return commit_from_source(ctx, src, n_cells * cell_size, cell_size, block_size, 0, 0, 0, true, true, out);
}

// ---- slot builder: a slot's blocks added in any order and in any number of pieces --------------------------------------
// The caller's bytes are copied into a ring of four pinned chunks (a quarter tile each); a chunk is copied to the device
// tile as soon as it is full, while the next one fills.  A full tile (tile_blocks blocks, the tile of hash_cells_staged) is
// hashed by the cell sponge, its block trees are built in a scratch forest and the results are scattered to their blocks'
// places in the handle: every forest level of a full handle, the block hashes of a compact one.  Two device tiles, each
// with its own compute stream, so that the kernels of one tile overlap the filling of the next.  Adds that do not complete
// a tile launch nothing.  The builder owns its streams and buffers: ctx->d_stage and ctx->h_pinned are shared with every
// other call on the context, so other calls may run between two adds.  The bookkeeping is in slot_builder.h.
#define CDX_BUILDER_CHUNKS 4

struct cdx_slot_builder {
  cdx_ctx* ctx = nullptr;
  cdx_slot* slot = nullptr;              // the handle being filled; a compact one has no forest below the block hashes
  SlotBuilderBook book;
  size_t cell_size = 0, block_size = 0, cpb = 0;
  size_t tile_blocks = 0, chunk_blocks = 0;
  uint64_t tiles = 0;                    // tiles flushed so far: the tile being filled goes to device tile tiles & 1
  size_t pos = 0;                        // blocks of the current tile in the pinned chunks
  size_t queued = 0;                     // ... of which the copy to the device tile has been queued
  int error = CDX_OK;                    // an earlier call failed on the device: the builder refuses everything after it
  std::vector<uint64_t> ids;             // the block at each position of the current tile
  cudaStream_t copy = nullptr, compute[2] = {nullptr, nullptr};
  cudaEvent_t ev_chunk[CDX_BUILDER_CHUNKS] = {};   // the last copy out of pinned chunk c
  cudaEvent_t ev_copied[2] = {}, ev_consumed[2] = {}, ev_join = nullptr;
  uint8_t* h_chunk[CDX_BUILDER_CHUNKS] = {};
  uint64_t* h_ids[2] = {nullptr, nullptr};         // pinned: the block-id table of device tile t on its way up
  DevBuf d_tile[2], d_ids[2], d_forest[2];
  std::vector<uint8_t*> forest[2];                 // the scratch forest's levels 0..block_depth, per device tile
};

static constexpr size_t kBuilderParallelFill = (size_t)4 << 20;   // pieces from this size on are copied by several host threads

// The builder's own streams, events and buffers, released in every state (the slot being built is not among them).
static void builder_release(cdx_slot_builder* b) {
  cudaSetDevice(b->ctx->device);
  for (cudaStream_t s : {b->copy, b->compute[0], b->compute[1]})
    if (s) cudaStreamSynchronize(s);
  for (int t = 0; t < 2; ++t)
    for (DevBuf* d : {&b->d_tile[t], &b->d_ids[t], &b->d_forest[t]}) {
      if (d->p) dev_free(d->p, d->st);
      d->p = nullptr;
    }
  for (int c = 0; c < CDX_BUILDER_CHUNKS; ++c) {
    if (b->h_chunk[c]) cudaFreeHost(b->h_chunk[c]);
    if (b->ev_chunk[c]) cudaEventDestroy(b->ev_chunk[c]);
    b->h_chunk[c] = nullptr;
    b->ev_chunk[c] = nullptr;
  }
  for (int t = 0; t < 2; ++t) {
    if (b->h_ids[t]) cudaFreeHost(b->h_ids[t]);
    if (b->ev_copied[t]) cudaEventDestroy(b->ev_copied[t]);
    if (b->ev_consumed[t]) cudaEventDestroy(b->ev_consumed[t]);
    b->h_ids[t] = nullptr;
    b->ev_copied[t] = b->ev_consumed[t] = nullptr;
    b->forest[t].clear();
  }
  if (b->ev_join) cudaEventDestroy(b->ev_join);
  b->ev_join = nullptr;
  for (cudaStream_t* s : {&b->copy, &b->compute[0], &b->compute[1]}) {
    if (*s) cudaStreamDestroy(*s);
    *s = nullptr;
  }
  std::vector<uint64_t>().swap(b->ids);
}

static int builder_setup(cdx_slot_builder* b, uint64_t n_blocks, bool compact) {
  cdx_ctx* ctx = b->ctx;
  size_t tile_blocks = (ctx->tile_mib << 20) / b->block_size;
  if (tile_blocks == 0) tile_blocks = 1;
  if (tile_blocks > n_blocks) tile_blocks = n_blocks;
  b->tile_blocks = tile_blocks;
  b->chunk_blocks = (tile_blocks + CDX_BUILDER_CHUNKS - 1) / CDX_BUILDER_CHUNKS;
  int rc = slot_alloc(ctx, n_blocks, b->cell_size, b->block_size, 0, n_blocks, 0, ctx->stream, &b->slot, false, compact);
  if (rc) return rc;
  try {
    slot_builder_init(&b->book, n_blocks);
    b->ids.assign(tile_blocks, 0);
  } catch (const std::bad_alloc&) {
    return fail(ctx, CDX_ERR_ALLOC, "host allocation of the bookkeeping of %llu blocks failed", (unsigned long long)n_blocks);
  }
  for (cudaStream_t* s : {&b->copy, &b->compute[0], &b->compute[1]}) CU_TRY(ctx, cudaStreamCreateWithFlags(s, cudaStreamNonBlocking));
  for (int c = 0; c < CDX_BUILDER_CHUNKS; ++c) CU_TRY(ctx, cudaEventCreateWithFlags(&b->ev_chunk[c], cudaEventDisableTiming));
  for (int t = 0; t < 2; ++t) {
    CU_TRY(ctx, cudaEventCreateWithFlags(&b->ev_copied[t], cudaEventDisableTiming));
    CU_TRY(ctx, cudaEventCreateWithFlags(&b->ev_consumed[t], cudaEventDisableTiming));
  }
  CU_TRY(ctx, cudaEventCreateWithFlags(&b->ev_join, cudaEventDisableTiming));
  // the handle's levels were allocated on ctx->stream, the builder's buffers are allocated on compute[0]
  CU_TRY(ctx, cudaEventRecord(b->ev_join, ctx->stream));
  CU_TRY(ctx, cudaStreamWaitEvent(b->compute[0], b->ev_join, 0));
  const size_t tile_cells = tile_blocks * b->cpb;
  const uint32_t bd = b->slot->block_depth;
  std::vector<size_t> f_off;
  size_t forest_nodes = 0;
  for (uint32_t l = 0; l <= bd; ++l) {
    f_off.push_back(forest_nodes);
    forest_nodes += b->cpb == 1 ? tile_cells : (tile_cells >> l);
  }
  for (int t = 0; t < 2; ++t) {
    if (b->d_tile[t].alloc(tile_blocks * b->block_size, b->compute[0]) != cudaSuccess || b->d_ids[t].alloc(8 * tile_blocks, b->compute[0]) != cudaSuccess ||
        b->d_forest[t].alloc(32 * forest_nodes, b->compute[0]) != cudaSuccess)
      return fail(ctx, CDX_ERR_ALLOC, "cudaMalloc of the slot builder's tiles failed");
    for (uint32_t l = 0; l <= bd; ++l) b->forest[t].push_back(b->d_forest[t].u8() + 32 * f_off[l]);
  }
  CU_TRY(ctx, cudaEventRecord(b->ev_join, b->compute[0]));
  CU_TRY(ctx, cudaStreamWaitEvent(b->copy, b->ev_join, 0));
  CU_TRY(ctx, cudaStreamWaitEvent(b->compute[1], b->ev_join, 0));
  const size_t n_chunks = (tile_blocks + b->chunk_blocks - 1) / b->chunk_blocks;
  for (size_t c = 0; c < n_chunks; ++c)
    if (cudaHostAlloc((void**)&b->h_chunk[c], b->chunk_blocks * b->block_size, cudaHostAllocDefault) != cudaSuccess)
      return fail(ctx, CDX_ERR_ALLOC, "cudaHostAlloc of %zu bytes failed", b->chunk_blocks * b->block_size);
  for (int t = 0; t < 2; ++t)
    if (cudaHostAlloc((void**)&b->h_ids[t], 8 * tile_blocks, cudaHostAllocDefault) != cudaSuccess)
      return fail(ctx, CDX_ERR_ALLOC, "cudaHostAlloc of %zu bytes failed", 8 * tile_blocks);
  return CDX_OK;
}

extern "C" int cdx_slot_builder_create(cdx_ctx* ctx, uint64_t n_blocks, size_t cell_size, size_t block_size, int keep_forest, cdx_slot_builder** out) {
  if (!ctx || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  char msg[160];
  int rc = slot_builder_shape(n_blocks, cell_size, block_size, msg, sizeof msg);
  if (rc) return fail(ctx, rc, "%s", msg);
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  cdx_slot_builder* b = new (std::nothrow) cdx_slot_builder();
  if (!b) return fail(ctx, CDX_ERR_ALLOC, "host allocation failed");
  b->ctx = ctx;
  b->cell_size = cell_size;
  b->block_size = block_size;
  b->cpb = block_size / cell_size;
  rc = builder_setup(b, n_blocks, keep_forest == 0);
  if (rc) {
    cdx_slot_builder_free(b);
    return rc;
  }
  *out = b;
  return CDX_OK;
}

// queue the copy of the pinned chunk being filled (blocks [queued, pos) of the current tile) to the device tile
static int builder_copy_chunk(cdx_slot_builder* b) {
  cdx_ctx* ctx = b->ctx;
  if (b->pos == b->queued) return CDX_OK;
  const int t = (int)(b->tiles & 1);
  if (b->queued == 0) CU_TRY(ctx, cudaStreamWaitEvent(b->copy, b->ev_consumed[t], 0));   // the tile before last is out of device tile t
  const size_t c = b->queued / b->chunk_blocks;
  CU_TRY(ctx, cudaMemcpyAsync(b->d_tile[t].u8() + b->queued * b->block_size, b->h_chunk[c], (b->pos - b->queued) * b->block_size,
                              cudaMemcpyHostToDevice, b->copy));
  CU_TRY(ctx, cudaEventRecord(b->ev_chunk[c], b->copy));
  b->queued = b->pos;
  return CDX_OK;
}

static int launch_scatter_felts(cdx_ctx* ctx, const uint8_t* src, const uint64_t* index, size_t n, uint8_t* dst, uint32_t width, cudaStream_t st) {
  k_scatter_felts<<<grid_for(2 * n * width, 256), 256, 0, st>>>(src, index, n, dst, width);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return CDX_OK;
}

// The current tile (pos blocks) through the cell sponge, its block trees and the scatter into the handle, on the compute
// stream of its device tile.
static int builder_flush(cdx_slot_builder* b) {
  cdx_ctx* ctx = b->ctx;
  cdx_slot* s = b->slot;
  int rc = builder_copy_chunk(b);
  if (rc) return rc;
  const int t = (int)(b->tiles & 1);
  const size_t nb = b->pos, n_cells = nb * b->cpb;
  const uint32_t bd = s->block_depth;
  CU_TRY(ctx, cudaEventSynchronize(b->ev_copied[t]));                 // the previous table uploaded from h_ids[t] has left it
  memcpy(b->h_ids[t], b->ids.data(), 8 * nb);
  CU_TRY(ctx, cudaMemcpyAsync(b->d_ids[t].p, b->h_ids[t], 8 * nb, cudaMemcpyHostToDevice, b->copy));
  CU_TRY(ctx, cudaEventRecord(b->ev_copied[t], b->copy));
  cudaStream_t cs = b->compute[t];
  CU_TRY(ctx, cudaStreamWaitEvent(cs, b->ev_copied[t], 0));
  rc = launch_hash_cells(ctx, b->d_tile[t].p, n_cells, b->cell_size, b->forest[t][0], cs);
  if (rc) return rc;
  rc = launch_block_trees(ctx, b->forest[t].data(), n_cells, b->cpb == 1, bd, cs);
  if (rc) return rc;
  const uint64_t* ids = (const uint64_t*)b->d_ids[t].p;
  if (s->compact) {
    rc = launch_scatter_felts(ctx, b->forest[t][bd], ids, nb, s->forest[bd], 1, cs);
    if (rc) return rc;
  } else {
    for (uint32_t l = 0; l <= bd; ++l) {                                // level l of block k: cpb >> l nodes from k * (cpb >> l)
      rc = launch_scatter_felts(ctx, b->forest[t][l], ids, nb, s->forest[l], b->cpb == 1 ? 1u : (uint32_t)(b->cpb >> l), cs);
      if (rc) return rc;
    }
  }
  CU_TRY(ctx, cudaEventRecord(b->ev_consumed[t], cs));
  ++b->tiles;
  b->pos = b->queued = 0;
  return CDX_OK;
}

// blocks [first, first + n) from data, already checked and marked
static int builder_take(cdx_slot_builder* b, uint64_t first, const uint8_t* data, uint64_t n) {
  cdx_ctx* ctx = b->ctx;
  const size_t bs = b->block_size;
  while (n) {
    const size_t c = b->pos / b->chunk_blocks, in = b->pos % b->chunk_blocks;
    const size_t chunk_end = std::min((c + 1) * b->chunk_blocks, b->tile_blocks);
    const size_t m = (size_t)std::min<uint64_t>(n, chunk_end - b->pos);
    if (in == 0) CU_TRY(ctx, cudaEventSynchronize(b->ev_chunk[c]));     // the chunk's last copy has left it (never recorded = done)
    uint8_t* dst = b->h_chunk[c] + in * bs;
    if (m * bs >= kBuilderParallelFill) {
      const ChunkFill fill = [data](uint8_t* d, uint64_t off, size_t len) { memcpy(d, data + off, len); };
      fill_chunk_parallel(fill, dst, 0, m * bs);
    } else {
      memcpy(dst, data, m * bs);
    }
    for (size_t k = 0; k < m; ++k) b->ids[b->pos + k] = first + k;
    b->pos += m;
    first += m;
    data += m * bs;
    n -= m;
    int rc = b->pos == chunk_end ? builder_copy_chunk(b) : CDX_OK;
    if (rc == CDX_OK && b->pos == b->tile_blocks) rc = builder_flush(b);
    if (rc) return rc;
  }
  return CDX_OK;
}

extern "C" int cdx_slot_builder_add_host(cdx_slot_builder* b, uint64_t first_block, const uint8_t* data, size_t n_bytes) {
  if (!b) return CDX_ERR_ARG;
  cdx_ctx* ctx = b->ctx;
  if (!data) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (b->error) return fail(ctx, CDX_ERR_STATE, "slot builder: an earlier call failed on the device, the builder cannot continue");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  char msg[160];
  uint64_t n = 0;
  int rc = slot_builder_add(&b->book, first_block, n_bytes, b->block_size, &n, msg, sizeof msg);
  if (rc) return fail(ctx, rc, "%s", msg);
  rc = builder_take(b, first_block, data, n);
  if (rc) b->error = rc;
  return rc;
}

extern "C" int cdx_slot_builder_finish(cdx_slot_builder* b, cdx_slot** out) {
  if (!b) return CDX_ERR_ARG;
  cdx_ctx* ctx = b->ctx;
  if (!out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  if (b->error) return fail(ctx, CDX_ERR_STATE, "slot builder: an earlier call failed on the device, the builder cannot continue");
  char msg[160];
  int rc = slot_builder_finish_status(&b->book, msg, sizeof msg);
  if (rc) return fail(ctx, rc, "%s", msg);
  cdx_slot* s = b->slot;
  auto body = [&]() -> int {
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (b->pos) {
      int r = builder_flush(b);
      if (r) return r;
    }
    for (int t = 0; t < 2; ++t) {                                       // the slot tree on the handle's stream, after both tiles
      CU_TRY(ctx, cudaEventRecord(b->ev_join, b->compute[t]));
      CU_TRY(ctx, cudaStreamWaitEvent(s->stream, b->ev_join, 0));
    }
    int r = build_top(s, s->low[0], true);
    if (r) return r;
    CU_TRY(ctx, cudaStreamSynchronize(s->stream));
    return CDX_OK;
  };
  rc = body();
  if (rc) {
    b->error = rc;
    return rc;
  }
  b->slot = nullptr;
  b->book.finished = true;
  std::vector<uint64_t>().swap(b->book.bits);
  builder_release(b);
  *out = s;
  return CDX_OK;
}

extern "C" void cdx_slot_builder_free(cdx_slot_builder* b) {
  if (!b) return;
  builder_release(b);
  if (b->slot) cdx_slot_free(b->slot);
  delete b;
}

// ---- persisted commitments ------------------------------------------------------------------------------------
// The image format and the header checks of import are in slot_image.h.

static size_t forest_node_count(const cdx_slot* s) {
  const uint64_t cpb = s->block_size / s->cell_size;
  if (s->compact) return s->n_local_blocks;
  size_t n = 0;
  for (uint32_t l = 0; l <= s->block_depth; ++l) n += cpb == 1 ? s->n_local_cells : (s->n_local_cells >> l);
  return n;
}
static size_t top_node_count(const cdx_slot* s) {   // slot levels 1..depth (level 0 is the forest's last layer)
  size_t n = 0;
  for (uint32_t l = 1; l <= s->slot_depth; ++l) n += s->width[l];
  return n;
}
static bool exportable(const cdx_slot* s) { return s && s->has_top && s->top_level == 0 && s->first_block == 0 && s->n_local_blocks == s->n_total_blocks; }

extern "C" size_t cdx_slot_export_size(const cdx_slot* s) {
  return exportable(s) ? sizeof(SlotImageHeader) + 32 * (forest_node_count(s) + top_node_count(s)) : 0;
}

extern "C" int cdx_slot_export(const cdx_slot* s, uint8_t* image, size_t image_bytes) {
  if (!s || !image) return CDX_ERR_ARG;
  cdx_ctx* ctx = s->ctx;
  if (!exportable(s)) return fail(ctx, CDX_ERR_STATE, "only whole slots with their top tree can be exported");
  if (image_bytes < cdx_slot_export_size(s)) return fail(ctx, CDX_ERR_SIZE, "image buffer too small");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  SlotImageHeader h;
  memset(&h, 0, sizeof h);
  memcpy(h.magic, s->compact ? "CDXSLOTC" : "CDXSLOT1", 8);
  h.cell_size = s->cell_size;
  h.block_size = s->block_size;
  h.n_blocks = s->n_total_blocks;
  h.forest_nodes = s->compact ? 0 : forest_node_count(s);
  h.top_nodes = top_node_count(s);
  h.block_depth = s->block_depth;
  h.slot_depth = s->slot_depth;
  memcpy(image, &h, sizeof h);
  uint8_t* p = image + sizeof h;
  if (s->compact) {
    CU_TRY(ctx, cudaMemcpyAsync(p, s->top[0], 32 * s->width[0], cudaMemcpyDeviceToHost, s->stream));
    p += 32 * s->width[0];
  } else {
    CU_TRY(ctx, cudaMemcpyAsync(p, s->d_forest, 32 * h.forest_nodes, cudaMemcpyDeviceToHost, s->stream));
    p += 32 * h.forest_nodes;
  }
  for (uint32_t l = 1; l <= s->slot_depth; ++l) {
    CU_TRY(ctx, cudaMemcpyAsync(p, s->top[l], 32 * s->width[l], cudaMemcpyDeviceToHost, s->stream));
    p += 32 * s->width[l];
  }
  CU_TRY(ctx, cudaStreamSynchronize(s->stream));
  return CDX_OK;
}

// The retained levels of an image that has just been copied to the device, checked in one launch of k_check_image: every
// stored parent against its stored children, every element canonical.  CDX_ERR_MISMATCH names the smallest bad node.
static int check_image_levels(cdx_slot* s) {
  cdx_ctx* ctx = s->ctx;
  ImageChain chain;
  memset(&chain, 0, sizeof chain);
  uint64_t total = 0;
  auto add = [&](const uint8_t* nodes, uint64_t n, uint32_t tree, uint32_t level, uint32_t bottom, uint32_t singles) {
    ImageLevel& L = chain.lv[chain.n_levels++];
    L = ImageLevel{nodes, n, total, (uint8_t)tree, (uint8_t)level, (uint8_t)bottom, (uint8_t)singles};
    total += n;
  };
  const bool singles = s->block_size / s->cell_size == 1;
  if (!s->compact)
    for (uint32_t l = 0; l <= s->block_depth; ++l) add(s->forest[l], singles ? s->n_local_cells : s->n_local_cells >> l, 0, l, l == 1, singles && l == 1);
  else
    add(s->top[0], s->width[0], 1, 0, 0, 0);
  for (uint32_t l = 1; l <= s->slot_depth; ++l) add(s->top[l], s->width[l], 1, l, l == 1, 0);
  DevBuf d_bad;
  CU_TRY(ctx, d_bad.alloc(8, s->stream));
  CU_TRY(ctx, cudaMemsetAsync(d_bad.p, 0xff, 8, s->stream));
  LAUNCH(ctx, k_check_image, total, s->stream, chain, total, (unsigned long long*)d_bad.p);
  unsigned long long bad = 0;
  CU_TRY(ctx, cudaMemcpyAsync(&bad, d_bad.p, 8, cudaMemcpyDeviceToHost, s->stream));
  CU_TRY(ctx, cudaStreamSynchronize(s->stream));
  if (bad == ~0ull) return CDX_OK;
  return fail(ctx, CDX_ERR_MISMATCH, "slot image: %s level %u node %llu %s", bad >> 63 ? "slot-tree" : "block-forest", (unsigned)(bad >> 57) & 63u,
              (bad & ((1ull << 57) - 1)) >> 1, bad & 1 ? "does not hash from its children" : "is not canonical");
}

extern "C" int cdx_slot_import(cdx_ctx* ctx, const uint8_t* image, size_t image_bytes, cdx_slot** out) {
  if (!ctx || !image || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  SlotImageLayout L;
  char msg[200];
  int rc = slot_image_layout(image, image_bytes, &L, msg, sizeof msg);
  if (rc) return fail(ctx, rc, "%s", msg);
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  cdx_slot* s = nullptr;
  rc = slot_alloc(ctx, L.n_blocks, L.cell_size, L.block_size, 0, L.n_blocks, 0, ctx->stream, &s, false, L.compact);
  if (rc) return rc;
  auto body = [&]() -> int {
    const uint8_t* p = image + sizeof(SlotImageHeader);
    CU_TRY(ctx, cudaMemcpyAsync(s->d_forest, p, 32 * L.level0_nodes, cudaMemcpyHostToDevice, s->stream));
    p += 32 * L.level0_nodes;
    CU_TRY(ctx, dev_alloc((void**)&s->d_top, 32 * L.top_nodes, s->stream));
    s->top.assign(s->slot_depth + 1, nullptr);
    s->top[0] = s->low[0];
    size_t off = 0;
    for (uint32_t l = 1; l <= s->slot_depth; ++l) {
      s->top[l] = s->d_top + 32 * off;
      off += s->width[l];
    }
    CU_TRY(ctx, cudaMemcpyAsync(s->d_top, p, 32 * L.top_nodes, cudaMemcpyHostToDevice, s->stream));
    s->top0_alias = true;
    s->has_top = true;
    return check_image_levels(s);
  };
  rc = body();
  if (rc) {
    cdx_slot_free(s);
    return rc;
  }
  *out = s;
  return CDX_OK;
}

// Release the block forest below the block hashes (SURVEY.md 8f.2: what a proof server keeps per slot).  Slot level 0 used
// to alias the end of d_forest; it moves into an allocation of its own, and d_forest is freed on the slot's stream.
extern "C" int cdx_slot_compact(cdx_slot* s) {
  if (!s) return CDX_ERR_ARG;
  cdx_ctx* ctx = s->ctx;
  if (!exportable(s)) return fail(ctx, CDX_ERR_STATE, "only whole slots with their top tree can be compacted");
  if (s->compact) return CDX_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  uint8_t* blocks = nullptr;
  const cudaError_t e = dev_alloc((void**)&blocks, 32 * s->n_local_blocks, s->stream);
  if (e != cudaSuccess) return fail(ctx, CDX_ERR_ALLOC, "cudaMalloc of %llu block hashes failed: %s", (unsigned long long)s->n_local_blocks, cudaGetErrorString(e));
  CU_TRY(ctx, cudaMemcpyAsync(blocks, s->forest[s->block_depth], 32 * s->n_local_blocks, cudaMemcpyDeviceToDevice, s->stream));
  dev_free(s->d_forest, s->stream);
  s->d_forest = blocks;
  for (uint32_t l = 0; l < s->block_depth; ++l) s->forest[l] = nullptr;
  s->forest[s->block_depth] = blocks;
  s->low[0] = blocks;
  if (s->top0_alias) s->top[0] = blocks;
  s->compact = true;
  CU_TRY(ctx, cudaStreamSynchronize(s->stream));
  return CDX_OK;
}

extern "C" size_t cdx_slot_device_bytes(const cdx_slot* s) {
  if (!s) return 0;
  size_t nodes = forest_node_count(s);
  for (uint32_t l = 1; l <= s->top_level; ++l) nodes += s->low_count[l];
  if (s->has_top)
    for (uint32_t l = s->top_level; l <= s->slot_depth; ++l)
      if (!(s->top0_alias && l == s->top_level)) nodes += s->width[l];
  return 32 * nodes;
}

extern "C" int cdx_slot_subtree_root_count(const cdx_slot* s, uint64_t* first_node, uint64_t* n_nodes) {
  if (!s) return CDX_ERR_ARG;
  if (first_node) *first_node = s->low_first[s->top_level];
  if (n_nodes) *n_nodes = s->low_count[s->top_level];
  return CDX_OK;
}

extern "C" const void* cdx_slot_subtree_roots_dev(const cdx_slot* s) { return s ? s->low[s->top_level] : nullptr; }

extern "C" int cdx_slot_subtree_roots_copy_dev(const cdx_slot* s, void* d_dst, void* stream) {
  if (!s || !d_dst) return CDX_ERR_ARG;
  cdx_ctx* ctx = s->ctx;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
  if (st != s->stream) CU_TRY(ctx, cudaStreamSynchronize(s->stream));
  CU_TRY(ctx, cudaMemcpyAsync(d_dst, s->low[s->top_level], 32 * s->low_count[s->top_level], cudaMemcpyDeviceToDevice, st));
  return CDX_OK;
}

extern "C" int cdx_slot_set_top_dev(cdx_slot* s, const void* d_level_nodes, uint64_t n_level_nodes, void* stream) {
  if (!s || !d_level_nodes) return CDX_ERR_ARG;
  cdx_ctx* ctx = s->ctx;
  if (n_level_nodes != s->width[s->top_level])
    return fail(ctx, CDX_ERR_SIZE, "expected %llu level-%u nodes, got %llu", (unsigned long long)s->width[s->top_level], s->top_level,
                (unsigned long long)n_level_nodes);
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (stream && (cudaStream_t)stream != s->stream) {   // order after everything queued on the old stream
    CU_TRY(ctx, cudaStreamSynchronize(s->stream));
    s->stream = (cudaStream_t)stream;
  }
  return build_top(s, (const uint8_t*)d_level_nodes, false);
}

extern "C" int cdx_slot_root(const cdx_slot* s, uint8_t root_out[32]) {
  if (!s || !root_out) return CDX_ERR_ARG;
  cdx_ctx* ctx = s->ctx;
  if (!s->has_top) return fail(ctx, CDX_ERR_STATE, "sharded slot has no top tree yet (call cdx_slot_set_top_dev)");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaMemcpyAsync(root_out, s->top[s->slot_depth], 32, cudaMemcpyDeviceToHost, s->stream));
  CU_TRY(ctx, cudaStreamSynchronize(s->stream));
  return CDX_OK;
}

extern "C" int cdx_slot_shape(const cdx_slot* s, uint64_t* n_cells, uint64_t* n_blocks, uint32_t* block_tree_depth, uint32_t* slot_tree_depth) {
  if (!s) return CDX_ERR_ARG;
  if (n_cells) *n_cells = s->n_total_blocks * (s->block_size / s->cell_size);
  if (n_blocks) *n_blocks = s->n_total_blocks;
  if (block_tree_depth) *block_tree_depth = s->block_depth;
  if (slot_tree_depth) *slot_tree_depth = s->slot_depth;
  return CDX_OK;
}

extern "C" int cdx_slot_read_layer(const cdx_slot* s, int tree, uint32_t level, uint64_t first, uint64_t count, uint8_t* out) {
  if (!s || !out) return CDX_ERR_ARG;
  cdx_ctx* ctx = s->ctx;
  if (count == 0) return CDX_OK;
  const uint8_t* src = nullptr;
  if (tree == 0) {
    if (level > s->block_depth) return fail(ctx, CDX_ERR_RANGE, "block-forest level %u > %u", level, s->block_depth);
    if (s->compact && level < s->block_depth)
      return fail(ctx, CDX_ERR_STATE, "the slot is compact: block-forest level %u was released (cdx_slot_prove_from_source rebuilds sampled blocks)", level);
    const uint64_t cpb = s->block_size / s->cell_size;
    const uint64_t per_block = cpb == 1 ? 1 : (cpb >> level);
    const uint64_t lo = s->first_block * per_block, n = s->n_local_blocks * per_block;
    if (first < lo || first + count > lo + n) return fail(ctx, CDX_ERR_RANGE, "nodes [%llu,+%llu) not held locally", (unsigned long long)first, (unsigned long long)count);
    src = s->forest[level] + 32 * (first - lo);
  } else if (tree == 1) {
    if (level > s->slot_depth) return fail(ctx, CDX_ERR_RANGE, "slot-tree level %u > %u", level, s->slot_depth);
    if (level >= s->top_level) {
      if (!s->has_top) return fail(ctx, CDX_ERR_STATE, "no top tree yet");
      if (first + count > s->width[level]) return fail(ctx, CDX_ERR_RANGE, "nodes out of range");
      src = s->top[level] + 32 * first;
    } else {
      if (first < s->low_first[level] || first + count > s->low_first[level] + s->low_count[level])
        return fail(ctx, CDX_ERR_RANGE, "nodes not held locally");
      src = s->low[level] + 32 * (first - s->low_first[level]);
    }
  } else {
    return fail(ctx, CDX_ERR_ARG, "tree must be 0 (block forest) or 1 (slot tree)");
  }
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaMemcpyAsync(out, src, 32 * count, cudaMemcpyDeviceToHost, s->stream));
  CU_TRY(ctx, cudaStreamSynchronize(s->stream));
  return CDX_OK;
}

static void make_path_plan(const cdx_slot* s, PathPlan& plan) {
  memset(&plan, 0, sizeof plan);
  plan.singles = (s->block_size / s->cell_size) == 1 ? 1u : 0u;
  for (uint32_t l = 0; l < s->block_depth; ++l) plan.forest[l] = s->forest[l];
  for (uint32_t l = 0; l <= s->slot_depth; ++l) {
    plan.width[l] = s->width[l];
    if (l >= s->top_level) plan.top[l] = s->top[l];
    else {
      plan.low[l] = s->low[l];
      plan.low_first[l] = s->low_first[l];
      plan.low_count[l] = s->low_count[l];
    }
  }
  plan.first_cell = s->first_block << s->cpb_log2;
  plan.n_local_cells = s->n_local_cells;
  plan.block_depth = s->block_depth;
  plan.slot_depth = s->slot_depth;
  plan.top_level = s->top_level;
  plan.cells_per_block_log2 = s->cpb_log2;
}

struct cdx_comm;
static int prove_core(const cdx_slot* s, cdx_comm* comm, const uint8_t* entropies, size_t n_challenges, size_t n_samples, const uint64_t* cells,
                      size_t max_depth, bool contribute_indices, uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out);   // capi_multi.cuh

extern "C" int cdx_slot_cell_paths(const cdx_slot* s, const uint64_t* cell_indices, size_t n_samples, size_t max_depth, uint8_t* out, uint8_t* leaf_out) {
  if (!s || !cell_indices || !out) return CDX_ERR_ARG;
  return prove_core(s, nullptr, nullptr, 0, n_samples, cell_indices, max_depth, true, nullptr, out, leaf_out);
}

// Proof-server call (SURVEY.md 8f.2): many challenges against one retained commitment.  Per challenge the reference
// runs cellIndices (sample/bn254.nim:26-27) and then one merkleProof pair per sample (gen_input/bn254.nim:53-74);
// here all challenges share three launches-worth of work: indices for every (challenge, counter) from the slot root
// that already lives on the device, the path gather reading those indices in place, one copy back.
extern "C" int cdx_slot_prove_batch(const cdx_slot* s, const uint8_t* entropies, size_t n_challenges, size_t n_samples, size_t max_depth,
                                    uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out) {
  if (!s || !entropies || !indices_out || !paths_out) return CDX_ERR_ARG;
  if (n_samples > 0xffffffffu) return fail(s->ctx, CDX_ERR_SIZE, "too many samples");
  return prove_core(s, nullptr, entropies, n_challenges, n_samples, nullptr, max_depth, true, indices_out, paths_out, leaves_out);
}

extern "C" int cdx_reconstruct_roots_host(cdx_ctx* ctx, const uint8_t* leaves, const uint64_t* indices, uint64_t n_leaves, const uint8_t* paths,
                                          size_t path_stride, size_t depth, size_t n, uint8_t* roots_out) {
  if (!ctx || !leaves || !indices || !roots_out || (!paths && depth)) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (depth > path_stride || depth > 64) return fail(ctx, CDX_ERR_RANGE, "depth %zu exceeds the path stride %zu", depth, path_stride);
  for (size_t i = 0; i < n; ++i)
    if (indices[i] >= n_leaves) return fail(ctx, CDX_ERR_RANGE, "leaf index %llu >= %llu", (unsigned long long)indices[i], (unsigned long long)n_leaves);
  if (n == 0) return CDX_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf dl, di, dp, dout;
  CU_TRY(ctx, dl.alloc(32 * n, ctx->stream));
  CU_TRY(ctx, di.alloc(8 * n, ctx->stream));
  CU_TRY(ctx, dp.alloc(32 * n * path_stride, ctx->stream));
  CU_TRY(ctx, dout.alloc(32 * n, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(dl.p, leaves, 32 * n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(di.p, indices, 8 * n, cudaMemcpyHostToDevice, ctx->stream));
  if (path_stride) CU_TRY(ctx, cudaMemcpyAsync(dp.p, paths, 32 * n * path_stride, cudaMemcpyHostToDevice, ctx->stream));
  LAUNCH(ctx, k_reconstruct_roots, n, ctx->stream, dl.u8(), (const uint64_t*)di.p, n_leaves, dp.u8(), (uint32_t)path_stride, (uint32_t)depth, n, dout.u8());
  CU_TRY(ctx, cudaMemcpyAsync(roots_out, dout.p, 32 * n, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

// ---- sampling and data source -------------------------------------------------------------------------------

extern "C" int cdx_cell_indices(cdx_ctx* ctx, const uint8_t entropy[32], const uint8_t slot_root[32], uint64_t n_cells, size_t n_samples, uint64_t* indices) {
  if (!ctx || !entropy || !slot_root || !indices) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (!is_pow2(n_cells)) return fail(ctx, CDX_ERR_NOT_POW2, "for this version, `numberOfCells` is assumed to be a power of two");
  if (n_samples == 0) return CDX_OK;
  if (n_samples > 0xffffffffu) return fail(ctx, CDX_ERR_SIZE, "too many samples");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf d_in, d_out;
  CU_TRY(ctx, d_in.alloc(64, ctx->stream));
  CU_TRY(ctx, d_out.alloc(8 * n_samples, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(d_in.p, entropy, 32, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(d_in.u8() + 32, slot_root, 32, cudaMemcpyHostToDevice, ctx->stream));
  LAUNCH(ctx, k_cell_indices, n_samples, ctx->stream, d_in.u8(), d_in.u8() + 32, n_cells - 1, (uint32_t)n_samples, n_samples, (uint64_t*)d_out.p);
  CU_TRY(ctx, cudaMemcpyAsync(indices, d_out.p, 8 * n_samples, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

static int launch_fake_cells(cdx_ctx* ctx, uint64_t seed, uint64_t first_cell, size_t n_cells, size_t cell_size, void* d_out, cudaStream_t st) {
  LAUNCH(ctx, k_fake_cells, n_cells, st, seed, first_cell, n_cells, (uint32_t)cell_size, (uint8_t*)d_out);
  return CDX_OK;
}

extern "C" int cdx_fake_cells_dev(cdx_ctx* ctx, uint64_t seed, uint64_t first_cell, size_t n_cells, size_t cell_size, void* d_out, void* stream) {
  if (!ctx || !d_out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (cell_size == 0 || cell_size % 4 || cell_size > (1u << 30)) return fail(ctx, CDX_ERR_SIZE, "cell size must be a non-zero multiple of 4");
  if (n_cells == 0) return CDX_OK;
  return launch_fake_cells(ctx, seed, first_cell, n_cells, cell_size, d_out, stream ? (cudaStream_t)stream : ctx->stream);
}

extern "C" int cdx_fake_cells_host(cdx_ctx* ctx, uint64_t seed, uint64_t first_cell, size_t n_cells, size_t cell_size, uint8_t* out) {
  if (!ctx || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (n_cells == 0) return CDX_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf d;
  CU_TRY(ctx, d.alloc(n_cells * cell_size, ctx->stream));
  int rc = cdx_fake_cells_dev(ctx, seed, first_cell, n_cells, cell_size, d.p, ctx->stream);
  if (rc) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(out, d.p, n_cells * cell_size, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

extern "C" int cdx_fill_synthetic_dev(cdx_ctx* ctx, uint64_t seed, uint64_t first_word, size_t n_bytes, void* d_out, void* stream) {
  if (!ctx || !d_out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (n_bytes % 8) return fail(ctx, CDX_ERR_SIZE, "synthetic fill needs a multiple of 8 bytes");
  if (n_bytes == 0) return CDX_OK;
  return launch_fill_synthetic(ctx, seed, first_word, n_bytes, d_out, stream ? (cudaStream_t)stream : ctx->stream);
}

static int launch_fill_synthetic(cdx_ctx* ctx, uint64_t seed, uint64_t first_word, size_t n_bytes, void* d_out, cudaStream_t st) {
  const size_t n_words = n_bytes / 8;
  size_t blocks = (n_words + 255) / 256;
  const size_t cap = (size_t)ctx->sm_count * 32;
  if (blocks > cap) blocks = cap;
  k_fill_synthetic<<<(unsigned)blocks, 256, 0, st>>>(seed, first_word, n_words, (uint64_t*)d_out);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return CDX_OK;
}

// Bytes [first_byte, first_byte + n_bytes) of a synthetic slot (include/codex_commit.h, CDX_SRC_SYNTHETIC) into d_out.
// Whole 8-byte words when the range and the destination allow it, else 4-byte halves: a slot of 100-byte blocks, a tile
// that starts inside a word, or a batch member behind a 300-byte one.  Cells are multiples of 4 bytes, so every range a
// slot, a tile or a batch asks for is 4-byte aligned.
static int fill_synthetic_range(cdx_ctx* ctx, uint64_t seed, uint64_t first_byte, size_t n_bytes, void* d_out, cudaStream_t st) {
  const uint64_t align = first_byte | n_bytes | (uintptr_t)d_out;
  if (align % 8 == 0) return launch_fill_synthetic(ctx, seed, first_byte / 8, n_bytes, d_out, st);
  if (align % 4) return fail(ctx, CDX_ERR_SIZE, "synthetic bytes [%llu,+%zu) are not 4-byte aligned", (unsigned long long)first_byte, n_bytes);
  const size_t n_halves = n_bytes / 4;
  size_t blocks = (n_halves + 255) / 256;
  const size_t cap = (size_t)ctx->sm_count * 32;
  if (blocks > cap) blocks = cap;
  k_fill_synthetic_halves<<<(unsigned)blocks, 256, 0, st>>>(seed, first_byte / 4, n_halves, (uint32_t*)d_out);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  return CDX_OK;
}

// ---- compact commitments: challenges answered from the slots' bytes ----------------------------------------------

static size_t prove_idx_region(size_t total);   // capi_multi.cuh

// The sampled forest holds the unique (slot, block) pairs of a call grouped by source class, then by the slot's first row,
// then by ascending block.  Each class reaches the cell sponge in one pass of the tile loop, whatever its number of slots.
enum { CLASS_FAKE = 0, CLASS_SYNTHETIC = 1, CLASS_READ = 2, N_CLASSES = 3 };

static uint32_t source_class(uint32_t kind) {
  return kind == CDX_SRC_FAKE ? CLASS_FAKE : kind == CDX_SRC_SYNTHETIC ? CLASS_SYNTHETIC : CLASS_READ;
}

// two descriptors of the same bytes: kind, size and the field the kind reads
static bool same_source(const cdx_slot_desc& a, const cdx_slot_desc& b) {
  if (a.kind != b.kind || a.n_bytes != b.n_bytes) return false;
  switch (a.kind) {
    case CDX_SRC_FAKE:
    case CDX_SRC_SYNTHETIC: return a.seed == b.seed;
    case CDX_SRC_FILE: return a.path == b.path || (a.path && b.path && strcmp(a.path, b.path) == 0);
    case CDX_SRC_HOST: return a.host == b.host;
    default: return true;                      // refused as an unknown kind
  }
}

struct SampledPairs {                          // the sampled forest's pairs, on the host and on the device
  std::vector<uint64_t> block;                 // pair j: block[j] of slot record slot[j]
  std::vector<uint32_t> slot;
  std::vector<const uint8_t*> host;            // per slot record: CDX_SRC_HOST bytes
  std::vector<const ChunkFill*> file;          // per slot record: CDX_SRC_FILE reader
  const uint64_t* d_block = nullptr;
  const uint32_t* d_slot = nullptr;
  const SampledSlot* d_slots = nullptr;
};

// The bytes of pairs [begin, begin + n), all of source class cls, through the tile loop: pair j lands in its tile at
// (j - begin - first) * block_size and its cell hashes at d_hashes + 32 * j * cpb; `consume` sees pair positions.
// Generated bytes take one k_generate_blocks launch per tile over the pairs on the device; host memory and files go
// through the pinned chunks, block by block.
static int hash_sampled_pairs(cdx_ctx* ctx, uint32_t cls, size_t begin, size_t n, const SampledPairs& P, size_t cell_size, size_t block_size,
                              uint8_t* d_hashes, const TileProducer* consume) {
  const size_t cpb = block_size / cell_size;
  uint8_t* hashes = d_hashes + 32 * begin * cpb;
  const TileProducer shifted = [&](int t, size_t first, size_t nb, uint8_t* tile, cudaStream_t cs) { return (*consume)(t, begin + first, nb, tile, cs); };
  const TileProducer* hook = consume ? &shifted : nullptr;
  if (cls != CLASS_READ) {
    size_t tile_blocks = (ctx->tile_mib << 20) / block_size;
    if (tile_blocks == 0) tile_blocks = 1;
    if (tile_blocks > n) tile_blocks = n;
    int rc = ensure_stage(ctx, tile_blocks * block_size);
    if (rc) return rc;
    const uint32_t fake = cls == CLASS_FAKE ? 1u : 0u;
    auto generate = [&](int, size_t first, size_t nb, uint8_t* dst, cudaStream_t st) -> int {
      const size_t units = nb * (fake ? block_size / cell_size : block_size / 4);   // cells or 4-byte halves
      size_t blocks = (units + 255) / 256;
      const size_t cap = (size_t)ctx->sm_count * 32;
      if (blocks > cap) blocks = cap;
      k_generate_blocks<<<(unsigned)blocks, 256, 0, st>>>(fake, P.d_slots, P.d_slot + begin + first, P.d_block + begin + first, nb,
                                                          (uint64_t)block_size, (uint32_t)cell_size, dst);
      ctx->launches++;
      CU_TRY(ctx, cudaGetLastError());
      return CDX_OK;
    };
    return run_tiles(ctx, tile_schedule(n, {}, tile_blocks), 2, nullptr, nullptr, cell_size, block_size, generate, hashes, hook);
  }
  ChunkFill fill = [&](uint8_t* dst, uint64_t off, size_t len) {   // pass offset -> the pair's bytes in its slot
    while (len) {
      const uint64_t j = begin + off / block_size, in = off % block_size;
      const size_t m = len < block_size - in ? len : (size_t)(block_size - in);
      const uint64_t at = P.block[j] * block_size + in;
      const uint32_t r = P.slot[j];
      if (P.host[r]) memcpy(dst, P.host[r] + at, m);
      else (*P.file[r])(dst, at, m);
      dst += m;
      off += m;
      len -= m;
    }
  };
  return hash_cells_staged(ctx, n * block_size, cell_size, block_size, fill, hashes, hook);
}

// cdx_slots_prove_from_source.  one_slot: cdx_slot_prove_from_source, where every row is slots[0] with sources[0] and the
// messages name no row.
static int prove_rows(const cdx_slot* const* slots, const cdx_slot_desc* sources, bool one_slot, const uint8_t* entropies, size_t n_rows,
                      size_t n_samples, size_t max_depth, uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out, uint8_t* cells_out) {
  cdx_ctx* ctx = slots[0]->ctx;
  if (!sources || !entropies || !indices_out || !paths_out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  char pre[48] = "";
  auto at = [&](size_t row) -> const char* {      // the message prefix naming a row
    if (!one_slot) snprintf(pre, sizeof pre, "challenge %zu: ", row);
    return pre;
  };
  // the distinct handles in the order of their first rows: slot record r is rec[r], first seen in row first_row[r]
  std::vector<const cdx_slot*> rec{slots[0]};
  std::vector<size_t> first_row{0};
  std::vector<uint32_t> row_slot;
  if (!one_slot) {
    row_slot.assign(n_rows, 0);
    std::unordered_map<const cdx_slot*, uint32_t> seen{{slots[0], 0u}};
    for (size_t k = 1; k < n_rows; ++k) {
      if (!slots[k]) return fail(ctx, CDX_ERR_ARG, "%snull slot", at(k));
      if (slots[k]->ctx != ctx) return fail(ctx, CDX_ERR_ARG, "%sthe slot belongs to another context than challenge 0's", at(k));
      const auto it = seen.emplace(slots[k], (uint32_t)rec.size());
      if (it.second) {
        rec.push_back(slots[k]);
        first_row.push_back(k);
      } else if (!same_source(sources[k], sources[first_row[it.first->second]])) {
        return fail(ctx, CDX_ERR_ARG, "%sthe slot's bytes are described differently in challenge %zu", at(k), first_row[it.first->second]);
      }
      row_slot[k] = it.first->second;
    }
  }
  const size_t n_rec = rec.size();
  auto src_of = [&](size_t r) -> const cdx_slot_desc& { return sources[one_slot ? 0 : first_row[r]]; };
  for (size_t r = 0; r < n_rec; ++r)
    if (!exportable(rec[r])) return fail(ctx, CDX_ERR_STATE, "%sonly whole slots with their top tree can be proven from their bytes", at(first_row[r]));
  if (n_samples > 0xffffffffu) return fail(ctx, CDX_ERR_SIZE, "too many samples");
  const size_t cell_size = rec[0]->cell_size, block_size = rec[0]->block_size, cpb = block_size / cell_size;
  const uint32_t cpb_log2 = rec[0]->cpb_log2, block_depth = rec[0]->block_depth;
  uint32_t deepest = 0;
  for (size_t r = 0; r < n_rec; ++r) {
    const cdx_slot* s = rec[r];
    if (s->cell_size != cell_size || s->block_size != block_size)
      return fail(ctx, CDX_ERR_SIZE, "%sslots of one call share one geometry: cells of %zu and blocks of %zu bytes here, %zu and %zu in challenge 0",
                  at(first_row[r]), s->cell_size, s->block_size, cell_size, block_size);
    if (src_of(r).n_bytes != s->n_total_blocks * block_size)
      return fail(ctx, CDX_ERR_SIZE, "%sthe source has %llu bytes, the slot %llu", at(first_row[r]), (unsigned long long)src_of(r).n_bytes,
                  (unsigned long long)(s->n_total_blocks * block_size));
    if (s->slot_depth > rec[deepest]->slot_depth) deepest = (uint32_t)r;
  }
  const cdx_slot* ds = rec[deepest];
  if (max_depth < ds->block_depth + ds->slot_depth || max_depth > 64)
    return fail(ctx, CDX_ERR_RANGE, "%smax_depth %zu < path length %u (padMerkleProof)", at(first_row[deepest]), max_depth, ds->block_depth + ds->slot_depth);
  if (ds->block_depth > 32 || ds->slot_depth >= 40) return fail(ctx, CDX_ERR_RANGE, "%stree too deep for the path plan", at(first_row[deepest]));
  const size_t total = n_rows * n_samples;
  if (total == 0) return CDX_OK;
  if (total > (1u << 20)) return fail(ctx, CDX_ERR_SIZE, "too many (challenge, sample) pairs in one call");
  if (one_slot) row_slot.assign(n_rows, 0);
  for (size_t r = 0; r < n_rec; ++r)
    if (!is_pow2(rec[r]->n_total_blocks << cpb_log2))
      return fail(ctx, CDX_ERR_NOT_POW2, "%sfor this version, `numberOfCells` is assumed to be a power of two", at(first_row[r]));
  // every source readable; files are opened before the pass
  std::vector<std::unique_ptr<FileSource>> files;
  SampledPairs P;
  P.host.assign(n_rec, nullptr);
  P.file.assign(n_rec, nullptr);
  std::vector<uint32_t> cls(n_rec);
  for (size_t r = 0; r < n_rec; ++r) {
    const cdx_slot_desc& d = src_of(r);
    switch (d.kind) {
      case CDX_SRC_FAKE:
      case CDX_SRC_SYNTHETIC: break;
      case CDX_SRC_HOST:
        if (!d.host) return fail(ctx, CDX_ERR_ARG, "%sslot descriptor without host pointer", at(first_row[r]));
        P.host[r] = d.host;
        break;
      case CDX_SRC_FILE:
        files.emplace_back(new FileSource);
        if (!d.path || !files.back()->open_path(d.path, 0))
          return fail(ctx, CDX_ERR_ARG, "%scannot open slot data file `%s`", at(first_row[r]), d.path ? d.path : "(null)");
        P.file[r] = &files.back()->fill;
        break;
      default: return fail(ctx, CDX_ERR_ARG, "%sunknown slot source kind %u", at(first_row[r]), d.kind);
    }
    cls[r] = source_class(d.kind);
  }
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  {                                                                                 // the retained levels are read on ctx->stream
    std::vector<cudaStream_t> synced{ctx->stream};
    for (const cdx_slot* s : rec)
      if (std::find(synced.begin(), synced.end(), s->stream) == synced.end()) {
        CU_TRY(ctx, cudaStreamSynchronize(s->stream));
        synced.push_back(s->stream);
      }
  }
  cudaStream_t st = ctx->stream;
  // [indices 8 B x total, padded to 16 B | paths 32 B x total x max_depth | leaves 32 B x total]: prove_core's layout
  const size_t idx_bytes = prove_idx_region(total), path_bytes = 32 * total * max_depth, leaf_bytes = 32 * total;
  DevBuf d_rows, d_all, d_tab, d_forest, d_cells, d_bad;
  auto body = [&]() -> int {
    // 1. per-row and per-slot tables: [entropies 32 B | root pointer 8 B | mask 8 B per row | slot records | slot levels |
    // row -> slot record 4 B per row]
    std::vector<SampledSlot> srec(n_rec);
    std::vector<SlotLevel> levels;
    for (size_t r = 0; r < n_rec; ++r) {
      const cdx_slot* s = rec[r];
      srec[r].seed = src_of(r).seed;
      srec[r].first_row = first_row[r];
      srec[r].levels = (uint32_t)levels.size();
      srec[r].slot_depth = s->slot_depth;
      for (uint32_t l = 0; l <= s->slot_depth; ++l) levels.push_back(SlotLevel{s->top[l], s->width[l]});
    }
    const size_t o_root = 32 * n_rows, o_mask = o_root + 8 * n_rows, o_slots = o_mask + 8 * n_rows;
    const size_t o_levels = o_slots + sizeof(SampledSlot) * n_rec, o_row_slot = o_levels + sizeof(SlotLevel) * levels.size();
    std::vector<uint8_t> rows(o_row_slot + 4 * n_rows);
    memcpy(rows.data(), entropies, 32 * n_rows);
    for (size_t k = 0; k < n_rows; ++k) {
      const cdx_slot* s = rec[row_slot[k]];
      const uint8_t* root = s->top[s->slot_depth];
      const uint64_t mask = (s->n_total_blocks << cpb_log2) - 1;
      memcpy(rows.data() + o_root + 8 * k, &root, 8);
      memcpy(rows.data() + o_mask + 8 * k, &mask, 8);
    }
    memcpy(rows.data() + o_slots, srec.data(), sizeof(SampledSlot) * n_rec);
    memcpy(rows.data() + o_levels, levels.data(), sizeof(SlotLevel) * levels.size());
    memcpy(rows.data() + o_row_slot, row_slot.data(), 4 * n_rows);
    int rc = upload_table(ctx, d_rows, rows.data(), rows.size(), st);
    if (rc) return rc;
    P.d_slots = (const SampledSlot*)(d_rows.u8() + o_slots);
    const SlotLevel* d_levels = (const SlotLevel*)(d_rows.u8() + o_levels);
    // 2. indices from the retained roots, copied back: the one host round trip
    CU_TRY(ctx, d_all.alloc(idx_bytes + path_bytes + leaf_bytes, st));
    const uint64_t* d_idx = (const uint64_t*)d_all.p;
    uint8_t* d_paths = d_all.u8() + idx_bytes;
    uint8_t* d_leaves = d_paths + path_bytes;
    LAUNCH(ctx, k_cell_indices_rows, total, st, d_rows.u8(), (const uint8_t* const*)(d_rows.u8() + o_root), (const uint64_t*)(d_rows.u8() + o_mask),
           (uint32_t)n_samples, total, (uint64_t*)d_all.p);
    CU_TRY(ctx, cudaMemcpyAsync(indices_out, d_idx, 8 * total, cudaMemcpyDeviceToHost, st));
    CU_TRY(ctx, cudaStreamSynchronize(st));
    // 3. the sampled forest's unique (slot, block) pairs (duplicate indices are normal, SURVEY.md Appendix C.4: each block is
    // read and hashed once), each sample's position among them, and the samples in the order of those positions
    std::vector<std::pair<uint64_t, uint64_t>> key(total), ukey;               // (class << 32 | slot record, block)
    for (size_t i = 0; i < total; ++i) {
      const uint32_t r = row_slot[i / n_samples];
      key[i] = {((uint64_t)cls[r] << 32) | r, indices_out[i] >> cpb_log2};
    }
    ukey = key;
    std::sort(ukey.begin(), ukey.end());
    ukey.erase(std::unique(ukey.begin(), ukey.end()), ukey.end());
    const size_t nu = ukey.size();
    P.block.resize(nu);
    P.slot.resize(nu);
    size_t class_begin[N_CLASSES + 1] = {0, 0, 0, 0};
    for (size_t j = 0; j < nu; ++j) {
      P.block[j] = ukey[j].second;
      P.slot[j] = (uint32_t)ukey[j].first;
      ++class_begin[(ukey[j].first >> 32) + 1];
    }
    for (int c = 0; c < N_CLASSES; ++c) class_begin[c + 1] += class_begin[c];
    std::vector<uint32_t> pos(total), order(total), first_sample(nu + 1, 0);   // samples of pair j: order[first_sample[j] ..)
    for (size_t i = 0; i < total; ++i) {
      pos[i] = (uint32_t)(std::lower_bound(ukey.begin(), ukey.end(), key[i]) - ukey.begin());
      ++first_sample[pos[i] + 1];
    }
    for (size_t j = 0; j < nu; ++j) first_sample[j + 1] += first_sample[j];
    {
      std::vector<uint32_t> next(first_sample.begin(), first_sample.end() - 1);
      for (size_t i = 0; i < total; ++i) order[next[pos[i]]++] = (uint32_t)i;
    }
    std::vector<uint8_t> tab(8 * nu + 8 * total + 4 * nu);                     // [pair blocks | pos | order | pair slot records]
    memcpy(tab.data(), P.block.data(), 8 * nu);
    memcpy(tab.data() + 8 * nu, pos.data(), 4 * total);
    memcpy(tab.data() + 8 * nu + 4 * total, order.data(), 4 * total);
    memcpy(tab.data() + 8 * nu + 8 * total, P.slot.data(), 4 * nu);
    rc = upload_table(ctx, d_tab, tab.data(), tab.size(), st);
    if (rc) return rc;
    P.d_block = (const uint64_t*)d_tab.p;
    const uint32_t* d_pos = (const uint32_t*)(d_tab.u8() + 8 * nu);
    const uint32_t* d_order = d_pos + total;
    P.d_slot = d_order + total;
    // 4-5. the sampled forest: the pairs' cell hashes, one tile pass per source class, then their block trees
    // (build_local_trees' rules)
    const size_t n_cells = nu * cpb;
    std::vector<size_t> f_off;
    size_t forest_nodes = 0;
    for (uint32_t l = 0; l <= block_depth; ++l) {
      f_off.push_back(forest_nodes);
      forest_nodes += cpb == 1 ? n_cells : (n_cells >> l);
    }
    CU_TRY(ctx, d_forest.alloc(32 * forest_nodes, st));
    std::vector<uint8_t*> forest;
    for (uint32_t l = 0; l <= block_depth; ++l) forest.push_back(d_forest.u8() + 32 * f_off[l]);
    if (cells_out) CU_TRY(ctx, d_cells.alloc(cell_size * total, st));
    // each sample's cell is copied out of its tile while the tile is resident (first: the tile's first pair)
    const TileProducer gather = [&](int, size_t first, size_t nb, uint8_t* tile, cudaStream_t cs) -> int {
      const size_t a = first_sample[first], n = first_sample[first + nb] - a, words = n * (cell_size / 4);
      if (n == 0) return CDX_OK;
      size_t blocks = (words + 255) / 256;
      const size_t cap = (size_t)ctx->sm_count * 32;
      if (blocks > cap) blocks = cap;
      k_gather_cells<<<(unsigned)blocks, 256, 0, cs>>>(tile, first, d_order + a, n, d_pos, d_idx, cpb_log2, (uint32_t)cell_size,
                                                        (uint64_t)block_size, d_cells.u8());
      ctx->launches++;
      CU_TRY(ctx, cudaGetLastError());
      return CDX_OK;
    };
    for (uint32_t c = 0; c < N_CLASSES; ++c) {
      if (class_begin[c + 1] == class_begin[c]) continue;
      rc = hash_sampled_pairs(ctx, c, class_begin[c], class_begin[c + 1] - class_begin[c], P, cell_size, block_size, forest[0],
                              cells_out ? &gather : nullptr);
      if (rc) return rc;
    }
    rc = launch_block_trees(ctx, forest.data(), n_cells, cpb == 1, block_depth, st);
    if (rc) return rc;
    // 6. every recomputed block hash against its slot's retained one
    CU_TRY(ctx, d_bad.alloc(8, st));
    CU_TRY(ctx, cudaMemsetAsync(d_bad.p, 0xff, 8, st));
    LAUNCH(ctx, k_check_sampled_blocks, nu, st, forest[block_depth], P.d_block, P.d_slot, nu, P.d_slots, d_levels, (unsigned long long*)d_bad.p);
    // 7. paths: block levels from the sampled forest, slot levels from each row's slot record
    SampledPathPlan plan;
    memset(&plan, 0, sizeof plan);
    for (uint32_t l = 0; l < block_depth; ++l) plan.forest[l] = forest[l];
    plan.row_slot = (const uint32_t*)(d_rows.u8() + o_row_slot);
    plan.slots = P.d_slots;
    plan.levels = d_levels;
    plan.block_depth = block_depth;
    plan.cells_per_block_log2 = cpb_log2;
    plan.n_samples = (uint32_t)n_samples;
    plan.singles = cpb == 1 ? 1u : 0u;
    const size_t threads = total * (max_depth + 1) * 2;
    k_gather_paths_sampled<<<grid_for(threads, 256), 256, 0, st>>>(plan, d_idx, d_pos, (uint32_t)total, (uint32_t)max_depth, d_paths, d_leaves);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    // 8. one copy back
    uint64_t bad = 0;
    CU_TRY(ctx, cudaMemcpyAsync(&bad, d_bad.p, 8, cudaMemcpyDeviceToHost, st));
    CU_TRY(ctx, cudaMemcpyAsync(paths_out, d_paths, path_bytes, cudaMemcpyDeviceToHost, st));
    if (leaves_out) CU_TRY(ctx, cudaMemcpyAsync(leaves_out, d_leaves, leaf_bytes, cudaMemcpyDeviceToHost, st));
    if (cells_out) CU_TRY(ctx, cudaMemcpyAsync(cells_out, d_cells.p, cell_size * total, cudaMemcpyDeviceToHost, st));
    CU_TRY(ctx, cudaStreamSynchronize(st));
    for (size_t r = 0, f = 0; r < n_rec; ++r)
      if (P.file[r] && files[f++]->io_errno.load())
        return fail(ctx, CDX_ERR_ARG, "%sreading slot data file `%s` failed: %s", at(first_row[r]), src_of(r).path, strerror(files[f - 1]->io_errno.load()));
    if (bad != UINT64_MAX)
      return fail(ctx, CDX_ERR_MISMATCH, "%sbytes of block %llu do not hash to the committed block hash", at(bad >> 44),
                  (unsigned long long)(bad & ((1ull << 44) - 1)));
    return CDX_OK;
  };
  const int rc = body();
  if (rc) drain_streams(ctx);
  return rc;
}

extern "C" int cdx_slot_prove_from_source(const cdx_slot* s, const cdx_slot_desc* source, const uint8_t* entropies, size_t n_challenges,
                                          size_t n_samples, size_t max_depth, uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out,
                                          uint8_t* cells_out) {
  if (!s) return CDX_ERR_ARG;
  return prove_rows(&s, source, true, entropies, n_challenges, n_samples, max_depth, indices_out, paths_out, leaves_out, cells_out);
}

extern "C" int cdx_slots_prove_from_source(const cdx_slot* const* slots, const cdx_slot_desc* sources, const uint8_t* entropies,
                                           size_t n_challenges, size_t n_samples, size_t max_depth, uint64_t* indices_out, uint8_t* paths_out,
                                           uint8_t* leaves_out, uint8_t* cells_out) {
  if (n_challenges == 0) return CDX_OK;
  if (!slots || !slots[0]) return CDX_ERR_ARG;
  return prove_rows(slots, sources, false, entropies, n_challenges, n_samples, max_depth, indices_out, paths_out, leaves_out, cells_out);
}

// ---- measurement --------------------------------------------------------------------------------------------

extern "C" int cdx_probe_imad_rate(cdx_ctx* ctx, int kind, double* ops_per_second, double* elapsed_ms) {
  if (!ctx || !ops_per_second) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (kind < 0 || kind > 2) return fail(ctx, CDX_ERR_ARG, "kind must be 0, 1 or 2");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf sink;
  CU_TRY(ctx, sink.alloc(4, ctx->stream));
  const unsigned blocks = (unsigned)ctx->sm_count * 8, threads = 256;
  const uint32_t iters = 8192;
  struct Events {                                   // destroyed on every exit path
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    ~Events() {
      if (e0) cudaEventDestroy(e0);
      if (e1) cudaEventDestroy(e1);
    }
  } ev;
  CU_TRY(ctx, cudaEventCreate(&ev.e0));
  CU_TRY(ctx, cudaEventCreate(&ev.e1));
  float best = 0.f;
  for (int rep = 0; rep < 4; ++rep) {   // rep 0 is the warm-up
    CU_TRY(ctx, cudaEventRecord(ev.e0, ctx->stream));
    k_probe_imad<<<blocks, threads, 0, ctx->stream>>>(kind, iters, 12345u + rep, (uint32_t*)sink.p);
    ctx->launches++;
    CU_TRY(ctx, cudaEventRecord(ev.e1, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    CU_TRY(ctx, cudaEventElapsedTime(&ms, ev.e0, ev.e1));
    if (rep > 0 && (best == 0.f || ms < best)) best = ms;
  }
  const double ops = (double)blocks * threads * iters * CDX_PROBE_OPS_PER_ITER;
  *ops_per_second = ops / (best * 1e-3);
  if (elapsed_ms) *elapsed_ms = best;
  return CDX_OK;
}

extern "C" int cdx_debug_guard_selftest(cdx_ctx* ctx) {
  if (!ctx) return CDX_ERR_ARG;
  if (!guard_enabled()) return fail(ctx, CDX_ERR_STATE, "CODEX_COMMIT_GUARD=1 is not set: nothing to test");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  {
    DevBuf d;
    CU_TRY(ctx, d.alloc(100, ctx->stream));
    CU_TRY(ctx, cudaMemsetAsync(d.u8() + 100, 0, 1, ctx->stream));   // one byte past the end, on purpose
  }                                                                  // ~DevBuf -> dev_free -> abort()
  return fail(ctx, CDX_ERR_STATE, "the guard band did not catch a deliberate overrun");
}

#include "capi_multi.cuh"
