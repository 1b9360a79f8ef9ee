// capi_multi.cuh -- second half of the C ABI (included at the end of capi.cu: one translation unit, because the kernels and
// their __constant__ / __device__ tables live in headers): batched small slots, NCCL communicators, block-range-sharded
// slots, dataset commitment and the all-GPUs-of-one-process group.  The reference does all of this in one sequential
// loop (reference/nim/proof_input/src/gen_input/bn254.nim:35-79); the entry points here are what a Nim host needs to run
// that loop on every GPU of a box through importc declarations alone.
#pragma once

#include <dlfcn.h>

#include <algorithm>
#include <mutex>
#include <numeric>
#include <string>

// ---- Merkle.digest over bytes -------------------------------------------------------------------------------------

// d_elems[k] = chunk k of the padded byte stream as a canonical field element (standard form, < 2^248)
__global__ void k_bytes_to_elements(const uint8_t* __restrict__ data, uint32_t len, uint32_t n_elems, uint8_t* __restrict__ out) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_elems) return;
  AnyBytes ld{data, len};
  st_felt(out + 32 * (size_t)k, read_chunk(ld, k));
}

extern "C" int cdx_merkle_root_bytes_host(cdx_ctx* ctx, const uint8_t* data, size_t len, uint8_t root_out[32]) {
  if (!ctx || !root_out || (!data && len)) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (len > 0x7fffffffu) return fail(ctx, CDX_ERR_SIZE, "byte string too long");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n = len / 31 + 1;                                              // Slot.hs:243-250
  const size_t total = cdx_merkle_total_nodes(n, 1);
  DevBuf d_bytes, d_tree;
  CU_TRY(ctx, d_bytes.alloc(len, ctx->stream));
  CU_TRY(ctx, d_tree.alloc(32 * total, ctx->stream));
  if (len) CU_TRY(ctx, cudaMemcpyAsync(d_bytes.p, data, len, cudaMemcpyHostToDevice, ctx->stream));
  LAUNCH(ctx, k_bytes_to_elements, n, ctx->stream, d_bytes.u8(), (uint32_t)len, (uint32_t)n, d_tree.u8());
  int rc = merkle_layers_on_device(ctx, d_tree.u8(), n, true, ctx->stream);
  if (rc) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(root_out, d_tree.u8() + 32 * (total - 1), 32, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

// ---- many small slots in one pass ---------------------------------------------------------------------------------

// Block forest over `n_cells` cell hashes at d_forest (levels concatenated: n_cells, n_cells/2, ..., n_blocks), then the slot
// trees of all slots at once; the slot roots land in d_roots (n_slots x 32 B).  Everything is queued on st.
static int batch_trees(cdx_ctx* ctx, uint8_t* d_forest, size_t n_cells, size_t cpb, const uint64_t* slot_blocks, size_t n_slots, uint8_t* d_roots,
                       cudaStream_t st, DevBuf& d_off, DevBuf& d_upper) {
  // block forest
  uint8_t* cur = d_forest;
  if (cpb == 1) {
    LAUNCH(ctx, k_merkle_level, n_cells, st, cur, n_cells, cur + 32 * n_cells, 1u, 1);
    cur += 32 * n_cells;
  } else {
    size_t n = n_cells;
    for (size_t w = cpb; w > 1; w >>= 1) {
      LAUNCH(ctx, k_merkle_level, n / 2, st, cur, n, cur + 32 * n, w == cpb ? 1u : 0u, 0);
      cur += 32 * n;
      n /= 2;
    }
  }
  // per-level widths and offsets of the slot trees (merkle/bn254.nim:29-60: n, ceil(n/2), ..., 1; a single block still
  // gets one key-3 compression)
  std::vector<std::vector<uint64_t>> off;
  std::vector<uint64_t> w(slot_blocks, slot_blocks + n_slots);
  for (int level = 0;; ++level) {
    std::vector<uint64_t> o(n_slots + 1, 0);
    for (size_t t = 0; t < n_slots; ++t) o[t + 1] = o[t] + w[t];
    const bool any = o[n_slots] != 0;
    off.push_back(std::move(o));
    if (!any) break;
    for (size_t t = 0; t < n_slots; ++t) w[t] = (level > 0 && w[t] <= 1) ? 0 : (w[t] + 1) / 2;
  }
  const size_t n_levels = off.size() - 1;            // off[n_levels] is all zero
  size_t upper_nodes = 0;
  for (size_t l = 1; l < n_levels; ++l) upper_nodes += off[l][n_slots];
  std::vector<uint64_t> flat;
  for (size_t l = 0; l < n_levels; ++l) flat.insert(flat.end(), off[l].begin(), off[l].end());
  CU_TRY(ctx, d_upper.alloc(32 * upper_nodes, st));
  {
    const int rc = upload_table(ctx, d_off, flat.data(), 8 * flat.size(), st);   // no stall of st: the sponge queued on it keeps running
    if (rc) return rc;
  }
  const uint64_t* offs = (const uint64_t*)d_off.p;
  const uint8_t* in = cur;                           // level 0 = the block hashes, last layer of the forest
  uint8_t* out = d_upper.u8();
  for (size_t l = 0; l + 1 < n_levels; ++l) {
    const size_t n_out = off[l + 1][n_slots];
    if (n_out > 0xffffffffull * CDX_BLOCK) return fail(ctx, CDX_ERR_SIZE, "batch too large");
    const unsigned blk = block_for(ctx, n_out);
    k_merkle_level_seg<<<grid_for(n_out, blk), blk, 0, st>>>(in, offs + l * (n_slots + 1), out, offs + (l + 1) * (n_slots + 1), (uint32_t)n_slots,
                                                              l == 0 ? 1u : 0u, d_roots);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    in = out;
    out += 32 * n_out;
  }
  return CDX_OK;
}

static size_t forest_nodes_for(size_t n_cells, size_t cpb) {
  if (cpb == 1) return 2 * n_cells;
  size_t total = 0;
  for (size_t n = n_cells, w = cpb;; n /= 2, w >>= 1) {
    total += n;
    if (w == 1) break;
  }
  return total;
}

static int check_batch(cdx_ctx* ctx, const uint64_t* slot_bytes, size_t n_slots, size_t cell_size, size_t block_size, size_t* total_bytes,
                       std::vector<uint64_t>& slot_blocks) {
  if (n_slots == 0 || n_slots > (1u << 24)) return fail(ctx, CDX_ERR_SIZE, "a batch holds 1 .. 2^24 slots");
  size_t total = 0;
  slot_blocks.resize(n_slots);
  for (size_t k = 0; k < n_slots; ++k) {
    int rc = check_shape(ctx, slot_bytes[k], cell_size, block_size);
    if (rc) return rc;
    slot_blocks[k] = slot_bytes[k] / block_size;
    total += slot_bytes[k];
  }
  *total_bytes = total;
  return CDX_OK;
}

// roots of a batch whose cell hashes are being produced into d_forest[0..n_cells) on st
static int batch_finish(cdx_ctx* ctx, DevBuf& d_forest, size_t n_cells, size_t cpb, const std::vector<uint64_t>& slot_blocks, cudaStream_t st,
                        uint8_t* roots_out_host, uint8_t* d_roots_out) {
  DevBuf d_off, d_upper, d_roots;
  uint8_t* d_r = d_roots_out;
  if (!d_r) {
    CU_TRY(ctx, d_roots.alloc(32 * slot_blocks.size(), st));
    d_r = d_roots.u8();
  }
  int rc = batch_trees(ctx, d_forest.u8(), n_cells, cpb, slot_blocks.data(), slot_blocks.size(), d_r, st, d_off, d_upper);
  if (rc) return rc;
  if (roots_out_host) {
    CU_TRY(ctx, cudaMemcpyAsync(roots_out_host, d_r, 32 * slot_blocks.size(), cudaMemcpyDeviceToHost, st));
    CU_TRY(ctx, cudaStreamSynchronize(st));
  }
  return CDX_OK;
}

extern "C" int cdx_slots_commit_batch_dev(cdx_ctx* ctx, const void* d_data, const uint64_t* slot_bytes, size_t n_slots, size_t cell_size,
                                          size_t block_size, void* stream, uint8_t* roots_out) {
  if (!ctx || !d_data || !slot_bytes || !roots_out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if ((uintptr_t)d_data % 16) return fail(ctx, CDX_ERR_ARG, "slot data must be 16-byte aligned");
  size_t total = 0;
  std::vector<uint64_t> slot_blocks;
  int rc = check_batch(ctx, slot_bytes, n_slots, cell_size, block_size, &total, slot_blocks);
  if (rc) return rc;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  const size_t n_cells = total / cell_size, cpb = block_size / cell_size;
  DevBuf d_forest;
  CU_TRY(ctx, d_forest.alloc(32 * forest_nodes_for(n_cells, cpb), st));
  rc = launch_hash_cells(ctx, d_data, n_cells, cell_size, d_forest.u8(), st);
  if (rc) return rc;
  return batch_finish(ctx, d_forest, n_cells, cpb, slot_blocks, st, roots_out, nullptr);
}

extern "C" int cdx_slots_commit_batch_host(cdx_ctx* ctx, const uint8_t* data, const uint64_t* slot_bytes, size_t n_slots, size_t cell_size,
                                           size_t block_size, uint8_t* roots_out) {
  if (!ctx || !data || !slot_bytes || !roots_out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  size_t total = 0;
  std::vector<uint64_t> slot_blocks;
  int rc = check_batch(ctx, slot_bytes, n_slots, cell_size, block_size, &total, slot_blocks);
  if (rc) return rc;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n_cells = total / cell_size, cpb = block_size / cell_size;
  DevBuf d_forest;
  CU_TRY(ctx, d_forest.alloc(32 * forest_nodes_for(n_cells, cpb), ctx->stream));
  rc = hash_cells_host(ctx, data, total, cell_size, block_size, d_forest.u8());   // the slots are contiguous: one stream of cells
  if (rc == CDX_OK) rc = batch_finish(ctx, d_forest, n_cells, cpb, slot_blocks, ctx->stream, roots_out, nullptr);
  if (rc) drain_streams(ctx);
  return rc;
}

extern "C" int cdx_slots_commit_batch_fake(cdx_ctx* ctx, const uint64_t* seeds, size_t n_slots, size_t n_cells_per_slot, size_t cell_size,
                                           size_t block_size, uint8_t* roots_out) {
  if (!ctx || !seeds || !roots_out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  if (cell_size == 0 || n_cells_per_slot == 0 || n_cells_per_slot > ((size_t)1 << 40) / cell_size) return fail(ctx, CDX_ERR_SIZE, "bad fake slot size");
  std::vector<uint64_t> slot_bytes(n_slots, (uint64_t)n_cells_per_slot * cell_size), slot_blocks;
  size_t total = 0;
  int rc = check_batch(ctx, slot_bytes.data(), n_slots, cell_size, block_size, &total, slot_blocks);
  if (rc) return rc;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t n_cells = total / cell_size, cpb = block_size / cell_size;
  DevBuf d_forest, d_data;
  CU_TRY(ctx, d_forest.alloc(32 * forest_nodes_for(n_cells, cpb), st));
  // the generator is sequential per cell and parallel across cells: one launch per slot, chunks of slots through one buffer
  const size_t chunk_slots = std::max<size_t>(1, ((size_t)1 << 30) / slot_bytes[0]);
  CU_TRY(ctx, d_data.alloc(std::min(chunk_slots, n_slots) * slot_bytes[0], st));
  for (size_t k0 = 0; k0 < n_slots; k0 += chunk_slots) {
    const size_t nk = std::min(chunk_slots, n_slots - k0);
    for (size_t k = 0; k < nk; ++k) {
      rc = launch_fake_cells(ctx, seeds[k0 + k], 0, n_cells_per_slot, cell_size, d_data.u8() + k * slot_bytes[0], st);
      if (rc) return rc;
    }
    rc = launch_hash_cells(ctx, d_data.p, nk * n_cells_per_slot, cell_size, d_forest.u8() + 32 * k0 * n_cells_per_slot, st);
    if (rc) return rc;
  }
  return batch_finish(ctx, d_forest, n_cells, cpb, slot_blocks, st, roots_out, nullptr);
}

// ---- NCCL, resolved at run time -----------------------------------------------------------------------------------

namespace {
struct NcclId {
  char internal[CDX_COMM_ID_BYTES];
};
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(NcclId*) = nullptr;
  int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  std::string error;
};
enum { kNcclUint8 = 1, kNcclSum = 0 };   // ncclDataType_t / ncclRedOp_t values (nccl.h; stable across 2.x)

NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* env = getenv("CODEX_COMMIT_NCCL_LIB");
    void* h = nullptr;
    if (env && *env) h = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // a copy that is already in the process (PyTorch's) wins
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
      api.error = std::string("libnccl.so.2 not found (set CODEX_COMMIT_NCCL_LIB): ") + (dlerror() ? dlerror() : "");
      return;
    }
    api.handle = h;
    api.GetUniqueId = (int (*)(NcclId*))dlsym(h, "ncclGetUniqueId");
    api.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(h, "ncclCommInitRank");
    api.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
    api.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(h, "ncclAllReduce");
    api.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
    if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllReduce || !api.GetErrorString) {
      api.error = "libnccl.so.2 lacks a required symbol";
      api.handle = nullptr;
    }
  });
  return &api;
}
}  // namespace

struct cdx_comm {
  cdx_ctx* ctx = nullptr;
  void* nccl = nullptr;      // ncclComm_t; null for a single rank
  int rank = 0, n_ranks = 1;
};

#define NCCL_TRY(ctx, call)                                                                                     \
  do {                                                                                                          \
    int _r = (call);                                                                                            \
    if (_r != 0) return fail((ctx), CDX_ERR_CUDA, "%s failed: %s", #call, nccl_api()->GetErrorString(_r));      \
  } while (0)

extern "C" int cdx_comm_unique_id(uint8_t id_out[CDX_COMM_ID_BYTES]) {
  if (!id_out) return CDX_ERR_ARG;
  NcclApi* api = nccl_api();
  if (!api->handle) return CDX_ERR_STATE;
  NcclId id;
  if (api->GetUniqueId(&id) != 0) return CDX_ERR_CUDA;
  memcpy(id_out, id.internal, CDX_COMM_ID_BYTES);
  return CDX_OK;
}

extern "C" int cdx_comm_init_rank(cdx_ctx* ctx, int n_ranks, int rank, const uint8_t id[CDX_COMM_ID_BYTES], cdx_comm** out) {
  if (!ctx || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(ctx, CDX_ERR_ARG, "rank %d outside 0..%d", rank, n_ranks - 1);
  cdx_comm* c = new (std::nothrow) cdx_comm();
  if (!c) return fail(ctx, CDX_ERR_ALLOC, "host allocation failed");
  c->ctx = ctx;
  c->rank = rank;
  c->n_ranks = n_ranks;
  if (n_ranks > 1) {
    NcclApi* api = nccl_api();
    if (!api->handle || !id) {
      delete c;
      return fail(ctx, CDX_ERR_STATE, "%s", !id ? "a communicator of several ranks needs the unique id" : api->error.c_str());
    }
    NcclId nid;
    memcpy(nid.internal, id, CDX_COMM_ID_BYTES);
    cudaError_t e = cudaSetDevice(ctx->device);
    const int r = e == cudaSuccess ? api->CommInitRank(&c->nccl, n_ranks, nid, rank) : -1;
    if (r != 0) {
      delete c;
      return fail(ctx, CDX_ERR_CUDA, "ncclCommInitRank failed: %s", r > 0 ? api->GetErrorString(r) : "cudaSetDevice");
    }
  }
  *out = c;
  return CDX_OK;
}

extern "C" void cdx_comm_destroy(cdx_comm* c) {
  if (!c) return;
  if (c->nccl) {
    cudaSetDevice(c->ctx->device);
    cudaStreamSynchronize(c->ctx->stream);
    nccl_api()->CommDestroy(c->nccl);
  }
  delete c;
}

extern "C" int cdx_comm_rank(const cdx_comm* c) { return c ? c->rank : 0; }
extern "C" int cdx_comm_size(const cdx_comm* c) { return c ? c->n_ranks : 1; }

// in-place byte-wise SUM over the ranks: every byte has at most one non-zero contributor on this path (disjoint block
// ranges, one owner per slot, one owner per sampled cell), so the sum is a gather/broadcast without per-rank counts
static int allreduce_bytes(cdx_ctx* ctx, cdx_comm* c, void* d_buf, size_t n_bytes, cudaStream_t st) {
  if (!c || c->n_ranks == 1 || n_bytes == 0) return CDX_OK;
  NCCL_TRY(ctx, nccl_api()->AllReduce(d_buf, d_buf, n_bytes, kNcclUint8, kNcclSum, c->nccl, st));
  return CDX_OK;
}

extern "C" int cdx_comm_barrier(cdx_comm* c) {
  if (!c) return CDX_ERR_ARG;
  cdx_ctx* ctx = c->ctx;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf d;
  CU_TRY(ctx, d.alloc(4, ctx->stream));
  CU_TRY(ctx, cudaMemsetAsync(d.p, 0, 4, ctx->stream));
  int rc = allreduce_bytes(ctx, c, d.p, 4, ctx->stream);
  if (rc) return rc;
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

// ---- block-range plans ----------------------------------------------------------------------------------------------

static uint64_t ceil_div_u64(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

extern "C" int cdx_plan_block_ranges(uint64_t n_total_blocks, int n_ranks, int* top_level, uint64_t* first_block, uint64_t* n_blocks) {
  if (n_total_blocks == 0 || n_ranks < 1 || !top_level || !first_block || !n_blocks) return CDX_ERR_ARG;
  // largest T whose 2^T-block chunks, dealt evenly, leave the heaviest rank within 1 % of the ideal share
  int t = 0;
  while (((uint64_t)1 << t) < n_total_blocks) ++t;
  int best = 0;
  for (; t > 0; --t) {
    const uint64_t n_chunks = ceil_div_u64(n_total_blocks, (uint64_t)1 << t);
    const uint64_t heaviest = std::min<uint64_t>(ceil_div_u64(n_chunks, (uint64_t)n_ranks) << t, n_total_blocks);
    if (n_chunks >= (uint64_t)n_ranks && (double)heaviest <= 1.01 * (double)n_total_blocks / n_ranks) {
      best = t;
      break;
    }
  }
  if (n_total_blocks == 1) best = 0;
  const uint64_t n_chunks = ceil_div_u64(n_total_blocks, (uint64_t)1 << best);
  for (int r = 0; r < n_ranks; ++r) {
    const uint64_t c0 = n_chunks * (uint64_t)r / n_ranks, c1 = n_chunks * (uint64_t)(r + 1) / n_ranks;
    const uint64_t b0 = std::min<uint64_t>(c0 << best, n_total_blocks), b1 = std::min<uint64_t>(c1 << best, n_total_blocks);
    first_block[r] = b0;
    n_blocks[r] = b1 - b0;
  }
  *top_level = best;
  return CDX_OK;
}

extern "C" int cdx_block_ranges_top_level(uint64_t n_total_blocks, int n_ranks, const uint64_t* first_block, const uint64_t* n_blocks, int* top_level) {
  if (n_total_blocks == 0 || n_ranks < 1 || !top_level || !first_block || !n_blocks) return CDX_ERR_ARG;
  uint64_t covered = 0;
  for (int r = 0; r < n_ranks; ++r) {
    if (n_blocks[r] && first_block[r] != covered) return CDX_ERR_RANGE;      // contiguous, in rank order
    covered += n_blocks[r];
  }
  if (covered != n_total_blocks) return CDX_ERR_RANGE;
  int depth = 0;                                                              // levels of the slot tree above the block hashes
  for (uint64_t w = n_total_blocks; w > 1; w = (w + 1) / 2) ++depth;
  int t = 0;
  for (; t < depth; ++t) {
    const uint64_t align = (uint64_t)1 << (t + 1);
    bool ok = true;
    for (int r = 0; r < n_ranks && ok; ++r) {
      if (n_blocks[r] == 0) continue;
      if (first_block[r] % align) ok = false;
      if (n_blocks[r] % align && first_block[r] + n_blocks[r] != n_total_blocks) ok = false;
    }
    if (!ok) break;
  }
  if (n_total_blocks == 1) t = 0;
  *top_level = t;
  return CDX_OK;
}

// ---- sharded slots ------------------------------------------------------------------------------------------------

extern "C" int cdx_slot_exchange_top(cdx_slot* s, cdx_comm* comm) {
  if (!s) return CDX_ERR_ARG;
  cdx_ctx* ctx = s->ctx;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const uint32_t T = s->top_level;
  const size_t W = s->width[T];
  DevBuf lvl;                                                                 // the complete level T, this rank's nodes in place, zeros elsewhere
  CU_TRY(ctx, lvl.alloc(32 * W, s->stream));
  CU_TRY(ctx, cudaMemsetAsync(lvl.p, 0, 32 * W, s->stream));
  if (s->low_count[T]) {
    if (s->low_first[T] + s->low_count[T] > W) return fail(ctx, CDX_ERR_RANGE, "local level-%u nodes exceed the level width", T);
    CU_TRY(ctx, cudaMemcpyAsync(lvl.u8() + 32 * s->low_first[T], s->low[T], 32 * s->low_count[T], cudaMemcpyDeviceToDevice, s->stream));
  }
  int rc = allreduce_bytes(ctx, comm, lvl.p, 32 * W, s->stream);
  if (rc) return rc;
  return build_top(s, lvl.u8(), false);                                       // copies the level, then the replicated upper levels
}

static int commit_sharded_common(cdx_ctx* ctx, cdx_comm* comm, const SlotSource& src, size_t n_local_bytes, size_t cell_size, size_t block_size,
                                 uint64_t first_block, uint64_t n_total_blocks, int top_level, bool sync, cdx_slot** out) {
  if (n_local_bytes) {
    int rc = check_shape(ctx, n_local_bytes, cell_size, block_size);
    if (rc) return rc;
  } else {
    int rc = check_shape(ctx, block_size, cell_size, block_size);
    if (rc) return rc;
  }
  cdx_slot* s = nullptr;
  int rc = commit_from_source(ctx, src, n_local_bytes, cell_size, block_size, first_block, n_total_blocks, top_level, false, false, &s);
  if (rc) return rc;
  rc = cdx_slot_exchange_top(s, comm);
  if (rc == CDX_OK && sync && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = fail(ctx, CDX_ERR_CUDA, "sharded commit failed on the device");
  if (rc) {
    drain_streams(ctx);
    cdx_slot_free(s);
    return rc;
  }
  *out = s;
  return CDX_OK;
}

extern "C" int cdx_slot_commit_sharded_host(cdx_ctx* ctx, cdx_comm* comm, const uint8_t* data, size_t n_local_bytes, size_t cell_size,
                                            size_t block_size, uint64_t first_block, uint64_t n_total_blocks, int top_level, cdx_slot** out) {
  if (!ctx || !out || (!data && n_local_bytes)) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  SlotSource src;
  src.kind = CDX_SRC_HOST;
  src.host = data;
  return commit_sharded_common(ctx, comm, src, n_local_bytes, cell_size, block_size, first_block, n_total_blocks, top_level, true, out);
}

extern "C" int cdx_slot_commit_sharded_dev(cdx_ctx* ctx, cdx_comm* comm, const void* d_data, size_t n_local_bytes, size_t cell_size, size_t block_size,
                                           uint64_t first_block, uint64_t n_total_blocks, int top_level, void* stream, cdx_slot** out) {
  if (!ctx || !out || (!d_data && n_local_bytes)) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  cdx_slot* s = nullptr;
  int rc;
  if (n_local_bytes) {
    rc = cdx_slot_commit_range_dev(ctx, d_data, n_local_bytes, cell_size, block_size, first_block, n_total_blocks, top_level, stream, &s);
  } else {
    rc = check_shape(ctx, block_size, cell_size, block_size);
    if (rc == CDX_OK) CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (rc == CDX_OK)
      rc = slot_alloc(ctx, 0, cell_size, block_size, first_block, n_total_blocks, top_level, stream ? (cudaStream_t)stream : ctx->stream, &s, true);
  }
  if (rc) return rc;
  rc = cdx_slot_exchange_top(s, comm);
  if (rc) {
    cudaStreamSynchronize(s->stream);
    cdx_slot_free(s);
    return rc;
  }
  *out = s;
  return CDX_OK;
}

// the gather kernel moves 16-byte halves: the paths must start 16-byte aligned behind the 8-byte indices
static size_t prove_idx_region(size_t total) { return (8 * total + 15) & ~(size_t)15; }

// cell indices (optional: from entropies) + path gather + optional byte-wise combine over the ranks + copy back.
//   d_entropies != null: indices for n_challenges x n_samples are derived on the device from the slot root;
//   otherwise `cells` (host) holds n_total indices.
// contribute_indices: whether this rank's copy of the indices takes part in the sum (exactly one rank's must).
static int prove_core(const cdx_slot* s, cdx_comm* comm, const uint8_t* entropies, size_t n_challenges, size_t n_samples, const uint64_t* cells,
                      size_t max_depth, bool contribute_indices, uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out) {
  cdx_ctx* ctx = s->ctx;
  if (s->compact) return fail(ctx, CDX_ERR_STATE, "the slot is compact: its block forest was released, answer challenges with cdx_slot_prove_from_source");
  if (!s->has_top) return fail(ctx, CDX_ERR_STATE, "no top tree yet");
  const uint64_t n_cells_total = s->n_total_blocks << s->cpb_log2;
  if (max_depth < s->block_depth + s->slot_depth || max_depth > 64)
    return fail(ctx, CDX_ERR_RANGE, "max_depth %zu < path length %u (padMerkleProof)", max_depth, s->block_depth + s->slot_depth);
  if (s->block_depth > 32 || s->slot_depth >= 40) return fail(ctx, CDX_ERR_RANGE, "tree too deep for the path plan");
  const size_t total = entropies ? n_challenges * n_samples : n_samples;
  if (total == 0) return CDX_OK;
  if (total > (1u << 20)) return fail(ctx, CDX_ERR_SIZE, "too many (challenge, sample) pairs in one call");
  if (entropies && !is_pow2(n_cells_total)) return fail(ctx, CDX_ERR_NOT_POW2, "for this version, `numberOfCells` is assumed to be a power of two");
  if (!entropies)
    for (size_t i = 0; i < total; ++i)
      if (cells[i] >= n_cells_total) return fail(ctx, CDX_ERR_RANGE, "cell index %llu >= %llu", (unsigned long long)cells[i], (unsigned long long)n_cells_total);
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  PathPlan plan;
  make_path_plan(s, plan);
  // one buffer: [indices 8 B x total, padded to 16 B | paths 32 B x total x max_depth | leaves 32 B x total]
  const size_t idx_bytes = prove_idx_region(total), path_bytes = 32 * total * max_depth, leaf_bytes = 32 * total;
  DevBuf d_ent, d_all;
  CU_TRY(ctx, d_all.alloc(idx_bytes + path_bytes + leaf_bytes, s->stream));
  uint64_t* d_idx = (uint64_t*)d_all.p;
  uint8_t* d_paths = d_all.u8() + idx_bytes;
  uint8_t* d_leaves = d_paths + path_bytes;
  if (entropies) {
    CU_TRY(ctx, d_ent.alloc(32 * n_challenges, s->stream));
    CU_TRY(ctx, cudaMemcpyAsync(d_ent.p, entropies, 32 * n_challenges, cudaMemcpyHostToDevice, s->stream));
    LAUNCH(ctx, k_cell_indices, total, s->stream, d_ent.u8(), (const uint8_t*)s->top[s->slot_depth], n_cells_total - 1, (uint32_t)n_samples, total, d_idx);
  } else {
    CU_TRY(ctx, cudaMemcpyAsync(d_idx, cells, 8 * total, cudaMemcpyHostToDevice, s->stream));
  }
  const size_t threads = total * (max_depth + 1) * 2;
  k_gather_paths<<<grid_for(threads, 256), 256, 0, s->stream>>>(plan, d_idx, (uint32_t)total, (uint32_t)max_depth, d_paths, d_leaves);
  ctx->launches++;
  CU_TRY(ctx, cudaGetLastError());
  if (comm && comm->n_ranks > 1) {
    if (!contribute_indices) CU_TRY(ctx, cudaMemsetAsync(d_idx, 0, idx_bytes, s->stream));
    int rc = allreduce_bytes(ctx, comm, d_all.p, idx_bytes + path_bytes + leaf_bytes, s->stream);
    if (rc) return rc;
  }
  if (indices_out) CU_TRY(ctx, cudaMemcpyAsync(indices_out, d_idx, 8 * total, cudaMemcpyDeviceToHost, s->stream));
  CU_TRY(ctx, cudaMemcpyAsync(paths_out, d_paths, path_bytes, cudaMemcpyDeviceToHost, s->stream));
  if (leaves_out) CU_TRY(ctx, cudaMemcpyAsync(leaves_out, d_leaves, leaf_bytes, cudaMemcpyDeviceToHost, s->stream));
  CU_TRY(ctx, cudaStreamSynchronize(s->stream));
  return CDX_OK;
}

extern "C" int cdx_slot_cell_paths_sharded(const cdx_slot* s, cdx_comm* comm, const uint64_t* cell_indices, size_t n_samples, size_t max_depth,
                                           uint8_t* out, uint8_t* leaf_out) {
  if (!s || !cell_indices || !out) return CDX_ERR_ARG;
  return prove_core(s, comm, nullptr, 0, n_samples, cell_indices, max_depth, !comm || comm->rank == 0, nullptr, out, leaf_out);
}

extern "C" int cdx_slot_prove_batch_sharded(const cdx_slot* s, cdx_comm* comm, const uint8_t* entropies, size_t n_challenges, size_t n_samples,
                                            size_t max_depth, uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out) {
  if (!s || !entropies || !indices_out || !paths_out) return CDX_ERR_ARG;
  if (n_samples > 0xffffffffu) return fail(s->ctx, CDX_ERR_SIZE, "too many samples");
  return prove_core(s, comm, entropies, n_challenges, n_samples, nullptr, max_depth, !comm || comm->rank == 0, indices_out, paths_out, leaves_out);
}

// ---- dataset commitment -------------------------------------------------------------------------------------------

struct cdx_dataset {
  cdx_ctx* ctx = nullptr;
  cdx_comm* comm = nullptr;
  size_t n_slots = 0, cell_size = 0, block_size = 0;
  std::vector<uint8_t> slot_roots;                 // n_slots x 32
  std::vector<std::vector<uint8_t>> layers;        // dataset tree, bottom first
  int64_t keep_slot = -1;
  cdx_slot* kept = nullptr;
  int kept_owner = -1;                             // rank holding the kept slot; -1: sharded over all ranks
  uint64_t kept_cells = 0;
  uint64_t bytes_local = 0;
  uint32_t n_whole = 0, n_batched = 0, n_sharded = 0;
};

namespace {
struct DatasetPlan {
  std::vector<int> owner;                          // per slot: rank, or -1 = sharded over all ranks
  std::vector<std::vector<size_t>> mine;           // per rank: its slots, largest first
};

// Slots are independent: longest-processing-time bin packing (largest slot first onto the least loaded rank).  A slot
// that alone would unbalance the ranks (more than a quarter of the ideal share, and at least 256 MiB per rank so the
// shards still fill a GPU) is block-range-sharded over all ranks instead.  Deterministic: every rank computes the same.
DatasetPlan plan_dataset(const std::vector<uint64_t>& blocks, int n_ranks, size_t block_size) {
  DatasetPlan p;
  const size_t n = blocks.size();
  p.owner.assign(n, 0);
  p.mine.assign(n_ranks, {});
  const uint64_t total = std::accumulate(blocks.begin(), blocks.end(), (uint64_t)0);
  const uint64_t min_shard_blocks = std::max<uint64_t>(1, ((uint64_t)256 << 20) / block_size) * (uint64_t)n_ranks;
  std::vector<size_t> order(n);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return blocks[a] > blocks[b]; });
  std::vector<uint64_t> load(n_ranks, 0);
  for (size_t k : order) {
    if (n_ranks > 1 && blocks[k] >= min_shard_blocks && blocks[k] * 4 * (uint64_t)n_ranks > total) {
      p.owner[k] = -1;
      continue;
    }
    const int r = (int)(std::min_element(load.begin(), load.end()) - load.begin());
    p.owner[k] = r;
    p.mine[r].push_back(k);
    load[r] += blocks[k];
  }
  return p;
}
}  // namespace

// bytes of one small slot into a device buffer (batches), queued on st
static int load_slot_bytes(cdx_ctx* ctx, const cdx_slot_desc& d, size_t cell_size, uint8_t* d_dst, cudaStream_t st, std::vector<std::vector<uint8_t>>& host_keep) {
  switch (d.kind) {
    case CDX_SRC_FAKE:
    case CDX_SRC_SYNTHETIC: return generate_bytes(ctx, d.kind, d.seed, 0, d.n_bytes, cell_size, d_dst, st);
    case CDX_SRC_HOST:
      if (!d.host) return fail(ctx, CDX_ERR_ARG, "slot descriptor without host pointer");
      CU_TRY(ctx, cudaMemcpyAsync(d_dst, d.host, d.n_bytes, cudaMemcpyHostToDevice, st));
      return CDX_OK;
    case CDX_SRC_FILE: {
      if (!d.path) return fail(ctx, CDX_ERR_ARG, "slot descriptor without path");
      FileSource f;
      if (!f.open_path(d.path, 0)) return fail(ctx, CDX_ERR_ARG, "cannot open slot data file `%s`", d.path);
      host_keep.emplace_back(d.n_bytes);
      f.fill(host_keep.back().data(), 0, d.n_bytes);
      if (f.io_errno.load()) return fail(ctx, CDX_ERR_ARG, "reading slot data file `%s` failed: %s", d.path, strerror(f.io_errno.load()));
      CU_TRY(ctx, cudaMemcpyAsync(d_dst, host_keep.back().data(), d.n_bytes, cudaMemcpyHostToDevice, st));
      return CDX_OK;
    }
    default: return fail(ctx, CDX_ERR_ARG, "unknown slot source kind %u", d.kind);
  }
}

// one slot (or this rank's block range of it) from its descriptor; no host synchronisation
static int commit_desc(cdx_ctx* ctx, cdx_comm* comm, const cdx_slot_desc& d, size_t cell_size, size_t block_size, bool sharded, cdx_slot** out) {
  const uint64_t n_total_blocks = d.n_bytes / block_size;
  uint64_t first = 0, count = n_total_blocks;
  int T = 0;
  if (sharded) {
    std::vector<uint64_t> f(comm->n_ranks), c(comm->n_ranks);
    int rc = cdx_plan_block_ranges(n_total_blocks, comm->n_ranks, &T, f.data(), c.data());
    if (rc) return fail(ctx, rc, "cannot plan block ranges");
    first = f[comm->rank];
    count = c[comm->rank];
  }
  SlotSource src;
  src.kind = d.kind;
  src.seed = d.seed;
  src.first_byte = first * block_size;
  FileSource file;
  if (d.kind == CDX_SRC_HOST) {
    if (!d.host) return fail(ctx, CDX_ERR_ARG, "slot descriptor without host pointer");
    src.host = d.host + first * block_size;
  } else if (d.kind == CDX_SRC_FILE) {
    if (!d.path || !file.open_path(d.path, first * block_size)) return fail(ctx, CDX_ERR_ARG, "cannot open slot data file `%s`", d.path ? d.path : "(null)");
    src.fill = &file.fill;
  } else if (d.kind != CDX_SRC_FAKE && d.kind != CDX_SRC_SYNTHETIC) {
    return fail(ctx, CDX_ERR_ARG, "unknown slot source kind %u", d.kind);
  }
  int rc;
  if (sharded) rc = commit_sharded_common(ctx, comm, src, count * block_size, cell_size, block_size, first, n_total_blocks, T, false, out);
  else rc = commit_from_source(ctx, src, d.n_bytes, cell_size, block_size, 0, 0, 0, true, false, out);
  if (rc == CDX_OK && file.io_errno.load()) {
    cudaStreamSynchronize(ctx->stream);
    cdx_slot_free(*out);
    *out = nullptr;
    return fail(ctx, CDX_ERR_ARG, "reading slot data file `%s` failed: %s", d.path, strerror(file.io_errno.load()));
  }
  return rc;
}

extern "C" int cdx_dataset_plan(const uint64_t* slot_bytes, size_t n_slots, size_t block_size, int n_ranks, int* owner_out) {
  if (!slot_bytes || !owner_out || n_slots == 0 || block_size == 0 || n_ranks < 1) return CDX_ERR_ARG;
  std::vector<uint64_t> blocks(n_slots);
  for (size_t k = 0; k < n_slots; ++k) {
    if (slot_bytes[k] == 0 || slot_bytes[k] % block_size) return CDX_ERR_SIZE;
    blocks[k] = slot_bytes[k] / block_size;
  }
  const DatasetPlan plan = plan_dataset(blocks, n_ranks, block_size);
  for (size_t k = 0; k < n_slots; ++k) owner_out[k] = plan.owner[k];
  return CDX_OK;
}

extern "C" void cdx_dataset_free(cdx_dataset* ds) {
  if (!ds) return;
  cdx_slot_free(ds->kept);
  delete ds;
}

extern "C" int cdx_dataset_commit(cdx_ctx* ctx, cdx_comm* comm, const cdx_slot_desc* slots, size_t n_slots, size_t cell_size, size_t block_size,
                                  int64_t keep_slot, cdx_dataset** out) {
  if (!ctx || !slots || !out) return fail(ctx, CDX_ERR_ARG, "null pointer");
  *out = nullptr;
  if (n_slots == 0 || n_slots > (1u << 24)) return fail(ctx, CDX_ERR_SIZE, "a dataset holds 1 .. 2^24 slots");
  if (keep_slot >= (int64_t)n_slots) return fail(ctx, CDX_ERR_RANGE, "keep_slot %lld outside the dataset", (long long)keep_slot);
  if (comm && comm->ctx != ctx) return fail(ctx, CDX_ERR_ARG, "the communicator belongs to another context");
  std::vector<uint64_t> blocks(n_slots);
  for (size_t k = 0; k < n_slots; ++k) {
    int rc = check_shape(ctx, slots[k].n_bytes, cell_size, block_size);
    if (rc) return rc;
    blocks[k] = slots[k].n_bytes / block_size;
  }
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const int n_ranks = comm ? comm->n_ranks : 1, rank = comm ? comm->rank : 0;
  const DatasetPlan plan = plan_dataset(blocks, n_ranks, block_size);
  cdx_dataset* ds = new (std::nothrow) cdx_dataset();
  if (!ds) return fail(ctx, CDX_ERR_ALLOC, "host allocation failed");
  ds->ctx = ctx;
  ds->comm = comm;
  ds->n_slots = n_slots;
  ds->cell_size = cell_size;
  ds->block_size = block_size;
  ds->keep_slot = keep_slot;
  const size_t cpb = block_size / cell_size;
  cudaStream_t st = ctx->stream;
  DevBuf d_roots;
  std::vector<std::vector<uint8_t>> host_keep;      // file bytes of batched slots, alive until the final synchronisation
  auto body = [&]() -> int {
    CU_TRY(ctx, d_roots.alloc(32 * n_slots, st));
    CU_TRY(ctx, cudaMemsetAsync(d_roots.p, 0, 32 * n_slots, st));
    auto take_root = [&](const cdx_slot* s, size_t k) -> int {
      CU_TRY(ctx, cudaMemcpyAsync(d_roots.u8() + 32 * k, s->top[s->slot_depth], 32, cudaMemcpyDeviceToDevice, st));
      return CDX_OK;
    };
    // 1. sharded slots, in index order (collective: every rank walks the same list)
    for (size_t k = 0; k < n_slots; ++k) {
      if (plan.owner[k] != -1) continue;
      cdx_slot* s = nullptr;
      int rc = commit_desc(ctx, comm, slots[k], cell_size, block_size, true, &s);
      if (rc) return rc;
      ds->bytes_local += s->n_local_blocks * block_size;
      ds->n_sharded++;
      if (rank == 0) rc = take_root(s, k);                                   // replicated: one contributor to the sum
      if ((int64_t)k == keep_slot) {
        ds->kept = s;
        ds->kept_owner = -1;
      } else {
        cdx_slot_free(s);                                                      // stream-ordered: frees after the queued work
      }
      if (rc) return rc;
    }
    // 2. this rank's own slots: big ones one by one, small ones (<= 64 MiB) in batches of up to 1 GiB
    const uint64_t small_bytes = (uint64_t)64 << 20, batch_cap = (uint64_t)1 << 30;
    std::vector<size_t> batch;
    uint64_t batch_bytes = 0;
    auto flush_batch = [&]() -> int {
      if (batch.empty()) return CDX_OK;
      DevBuf d_data, d_forest, d_batch_roots;
      CU_TRY(ctx, d_data.alloc(batch_bytes, st));
      const size_t n_cells = batch_bytes / cell_size;
      CU_TRY(ctx, d_forest.alloc(32 * forest_nodes_for(n_cells, cpb), st));
      CU_TRY(ctx, d_batch_roots.alloc(32 * batch.size(), st));
      std::vector<uint64_t> bb;
      uint64_t off = 0;
      for (size_t k : batch) {
        int rc = load_slot_bytes(ctx, slots[k], cell_size, d_data.u8() + off, st, host_keep);
        if (rc) return rc;
        off += slots[k].n_bytes;
        bb.push_back(blocks[k]);
      }
      int rc = launch_hash_cells(ctx, d_data.p, n_cells, cell_size, d_forest.u8(), st);
      if (rc) return rc;
      rc = batch_finish(ctx, d_forest, n_cells, cpb, bb, st, nullptr, d_batch_roots.u8());
      if (rc) return rc;
      {                                                                        // batch roots into their places: one launch, not one copy per slot
        std::vector<uint64_t> where(batch.begin(), batch.end());
        DevBuf d_where;
        rc = upload_table(ctx, d_where, where.data(), 8 * where.size(), st);
        if (rc) return rc;
        k_scatter_felts<<<grid_for(2 * where.size(), 256), 256, 0, st>>>(d_batch_roots.u8(), (const uint64_t*)d_where.p, where.size(), d_roots.u8());
        ctx->launches++;
        CU_TRY(ctx, cudaGetLastError());
      }
      ds->n_batched += (uint32_t)batch.size();
      ds->bytes_local += batch_bytes;
      batch.clear();
      batch_bytes = 0;
      return CDX_OK;
    };
    for (size_t k : plan.mine[rank]) {
      const bool keep = (int64_t)k == keep_slot;
      if (!keep && slots[k].n_bytes <= small_bytes) {
        if (batch_bytes + slots[k].n_bytes > batch_cap) {
          int rc = flush_batch();
          if (rc) return rc;
        }
        batch.push_back(k);
        batch_bytes += slots[k].n_bytes;
        continue;
      }
      cdx_slot* s = nullptr;
      int rc = commit_desc(ctx, comm, slots[k], cell_size, block_size, false, &s);
      if (rc) return rc;
      ds->bytes_local += slots[k].n_bytes;
      ds->n_whole++;
      rc = take_root(s, k);
      if (keep) {
        ds->kept = s;
        ds->kept_owner = rank;
      } else {
        cdx_slot_free(s);
      }
      if (rc) return rc;
    }
    int rc = flush_batch();
    if (rc) return rc;
    // 3. one collective for all slot roots, then the dataset tree on every rank (gen_input/bn254.nim:49)
    rc = allreduce_bytes(ctx, comm, d_roots.p, 32 * n_slots, st);
    if (rc) return rc;
    const size_t total = cdx_merkle_total_nodes(n_slots, 1);
    DevBuf d_tree;
    CU_TRY(ctx, d_tree.alloc(32 * total, st));
    CU_TRY(ctx, cudaMemcpyAsync(d_tree.p, d_roots.p, 32 * n_slots, cudaMemcpyDeviceToDevice, st));
    rc = merkle_layers_on_device(ctx, d_tree.u8(), n_slots, true, st);
    if (rc) return rc;
    std::vector<uint8_t> flat(32 * total);
    CU_TRY(ctx, cudaMemcpyAsync(flat.data(), d_tree.p, 32 * total, cudaMemcpyDeviceToHost, st));
    CU_TRY(ctx, cudaStreamSynchronize(st));
    size_t off = 0, m = n_slots;
    const int n_layers = cdx_merkle_num_layers(n_slots, 1);
    for (int l = 0; l < n_layers; ++l) {
      ds->layers.emplace_back(flat.begin() + 32 * off, flat.begin() + 32 * (off + m));
      off += m;
      m = (m + 1) / 2;
    }
    ds->slot_roots = ds->layers[0];
    if (keep_slot >= 0) {
      ds->kept_cells = blocks[(size_t)keep_slot] * cpb;
      if (plan.owner[(size_t)keep_slot] >= 0) ds->kept_owner = plan.owner[(size_t)keep_slot];
    }
    return CDX_OK;
  };
  const int rc = body();
  if (rc) {
    drain_streams(ctx);
    cdx_dataset_free(ds);
    return rc;
  }
  *out = ds;
  return CDX_OK;
}

extern "C" int cdx_dataset_root(const cdx_dataset* ds, uint8_t root_out[32]) {
  if (!ds || !root_out || ds->layers.empty()) return CDX_ERR_ARG;
  memcpy(root_out, ds->layers.back().data(), 32);
  return CDX_OK;
}

extern "C" int cdx_dataset_slot_roots(const cdx_dataset* ds, uint8_t* roots_out) {
  if (!ds || !roots_out) return CDX_ERR_ARG;
  memcpy(roots_out, ds->slot_roots.data(), ds->slot_roots.size());
  return CDX_OK;
}

extern "C" int cdx_dataset_slot_proof(const cdx_dataset* ds, uint64_t slot_index, size_t max_log2_nslots, uint8_t* path_out) {
  if (!ds || !path_out) return CDX_ERR_ARG;
  cdx_ctx* ctx = ds->ctx;
  if (slot_index >= ds->n_slots) return fail(ctx, CDX_ERR_RANGE, "slot index %llu outside the dataset", (unsigned long long)slot_index);
  const size_t depth = ds->layers.size() - 1;
  if (depth > max_log2_nslots) return fail(ctx, CDX_ERR_RANGE, "dataset tree depth %zu exceeds maxLog2NSlots %zu (padMerkleProof)", depth, max_log2_nslots);
  memset(path_out, 0, 32 * max_log2_nslots);
  uint64_t k = slot_index, m = ds->n_slots;                                   // merkleProof: merkle.nim:21-42
  for (size_t i = 0; i < depth; ++i) {
    const uint64_t j = k ^ 1;
    if (j < m) memcpy(path_out + 32 * i, ds->layers[i].data() + 32 * j, 32);
    k >>= 1;
    m = (m + 1) >> 1;
  }
  return CDX_OK;
}

extern "C" int cdx_dataset_stats(const cdx_dataset* ds, uint64_t* bytes_local, uint32_t* n_whole, uint32_t* n_batched, uint32_t* n_sharded) {
  if (!ds) return CDX_ERR_ARG;
  if (bytes_local) *bytes_local = ds->bytes_local;
  if (n_whole) *n_whole = ds->n_whole;
  if (n_batched) *n_batched = ds->n_batched;
  if (n_sharded) *n_sharded = ds->n_sharded;
  return CDX_OK;
}

extern "C" cdx_slot* cdx_dataset_kept_slot(const cdx_dataset* ds) { return ds ? ds->kept : nullptr; }

extern "C" int cdx_dataset_prove(const cdx_dataset* ds, const uint8_t entropy[32], size_t n_samples, size_t max_depth, uint64_t* indices_out,
                                 uint8_t* paths_out, uint8_t* leaves_out) {
  if (!ds || !entropy || !indices_out || !paths_out) return CDX_ERR_ARG;
  cdx_ctx* ctx = ds->ctx;
  if (ds->keep_slot < 0) return fail(ctx, CDX_ERR_STATE, "the dataset was committed without a kept slot");
  if (n_samples == 0) return CDX_OK;
  if (n_samples > (1u << 20)) return fail(ctx, CDX_ERR_SIZE, "too many samples");
  if (!is_pow2(ds->kept_cells)) return fail(ctx, CDX_ERR_NOT_POW2, "for this version, `numberOfCells` is assumed to be a power of two");
  const int rank = ds->comm ? ds->comm->rank : 0;
  if (ds->kept_owner == -1 || ds->kept_owner == rank) {
    if (!ds->kept) return fail(ctx, CDX_ERR_STATE, "the kept slot is missing on its owner");
    // sharded: every rank gathers its part, rank 0 contributes the indices; whole: the owner contributes everything
    const bool idx = ds->kept_owner == rank || rank == 0;
    return prove_core(ds->kept, ds->comm, entropy, 1, n_samples, nullptr, max_depth, idx, indices_out, paths_out, leaves_out);
  }
  // not the owner: contribute zeros to the same collective and receive the answer
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t idx_bytes = prove_idx_region(n_samples);               // the owner's layout (prove_core)
  const size_t bytes = idx_bytes + 32 * n_samples * max_depth + 32 * n_samples;
  DevBuf d;
  CU_TRY(ctx, d.alloc(bytes, ctx->stream));
  CU_TRY(ctx, cudaMemsetAsync(d.p, 0, bytes, ctx->stream));
  int rc = allreduce_bytes(ctx, ds->comm, d.p, bytes, ctx->stream);
  if (rc) return rc;
  CU_TRY(ctx, cudaMemcpyAsync(indices_out, d.p, 8 * n_samples, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaMemcpyAsync(paths_out, d.u8() + idx_bytes, 32 * n_samples * max_depth, cudaMemcpyDeviceToHost, ctx->stream));
  if (leaves_out) CU_TRY(ctx, cudaMemcpyAsync(leaves_out, d.u8() + idx_bytes + 32 * n_samples * max_depth, 32 * n_samples, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return CDX_OK;
}

// ---- all GPUs of one process --------------------------------------------------------------------------------------

struct cdx_group {
  std::vector<cdx_ctx*> ctx;
  std::vector<cdx_comm*> comm;
  std::string err;
};

namespace {
// fn(rank) on one thread per GPU; returns the first non-zero status and records that rank's message
template <class Fn>
int group_run(cdx_group* g, Fn fn) {
  const int n = (int)g->ctx.size();
  std::vector<int> rc(n, CDX_OK);
  if (n == 1) {
    rc[0] = fn(0);
  } else {
    std::vector<std::thread> thr;
    for (int r = 0; r < n; ++r) thr.emplace_back([&, r]() { rc[r] = fn(r); });
    for (auto& t : thr) t.join();
  }
  for (int r = 0; r < n; ++r)
    if (rc[r] != CDX_OK) {
      g->err = "rank " + std::to_string(r) + ": " + cdx_last_error(g->ctx[r]);
      return rc[r];
    }
  return CDX_OK;
}
}  // namespace

extern "C" void cdx_group_destroy(cdx_group* g) {
  if (!g) return;
  for (cdx_comm* c : g->comm) cdx_comm_destroy(c);
  for (cdx_ctx* c : g->ctx) cdx_ctx_destroy(c);
  delete g;
}

extern "C" int cdx_group_create(const int* devices, int n_devices, cdx_group** out) {
  if (!out) return CDX_ERR_ARG;
  *out = nullptr;
  std::vector<int> devs;
  if (devices && n_devices > 0) {
    devs.assign(devices, devices + n_devices);
  } else {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return CDX_ERR_CUDA;
    for (int i = 0; i < n; ++i) devs.push_back(i);
  }
  cdx_group* g = new (std::nothrow) cdx_group();
  if (!g) return CDX_ERR_ALLOC;
  // one CUDA primary context per device: created in parallel, it is most of the group's start-up time
  g->ctx.assign(devs.size(), nullptr);
  {
    std::vector<int> rcs(devs.size(), CDX_OK);
    std::vector<std::thread> thr;
    for (size_t r = 0; r < devs.size(); ++r) thr.emplace_back([&, r]() { rcs[r] = cdx_ctx_create(devs[r], &g->ctx[r]); });
    for (auto& t : thr) t.join();
    for (size_t r = 0; r < devs.size(); ++r)
      if (rcs[r] != CDX_OK) {
        const int rc = rcs[r];
        cdx_group_destroy(g);
        return rc;
      }
  }
  const int n = (int)devs.size();
  g->comm.assign(n, nullptr);
  uint8_t id[CDX_COMM_ID_BYTES] = {0};
  if (n > 1) {
    const int rc = cdx_comm_unique_id(id);
    if (rc) {
      cdx_group_destroy(g);
      return rc;
    }
  }
  const int rc = group_run(g, [&](int r) { return cdx_comm_init_rank(g->ctx[r], n, r, id, &g->comm[r]); });
  if (rc) {
    cdx_group_destroy(g);
    return rc;
  }
  *out = g;
  return CDX_OK;
}

extern "C" int cdx_group_size(const cdx_group* g) { return g ? (int)g->ctx.size() : 0; }
extern "C" cdx_ctx* cdx_group_ctx(const cdx_group* g, int rank) { return g && rank >= 0 && rank < (int)g->ctx.size() ? g->ctx[rank] : nullptr; }
extern "C" cdx_comm* cdx_group_comm(const cdx_group* g, int rank) { return g && rank >= 0 && rank < (int)g->comm.size() ? g->comm[rank] : nullptr; }
extern "C" const char* cdx_group_last_error(const cdx_group* g) { return g ? g->err.c_str() : "no group"; }

extern "C" int cdx_group_slot_commit_host(cdx_group* g, const uint8_t* data, size_t n_bytes, size_t cell_size, size_t block_size, cdx_slot** slots_out) {
  if (!g || !data || !slots_out) return CDX_ERR_ARG;
  const int n = (int)g->ctx.size();
  for (int r = 0; r < n; ++r) slots_out[r] = nullptr;
  int rc = check_shape(g->ctx[0], n_bytes, cell_size, block_size);
  if (rc) {
    g->err = cdx_last_error(g->ctx[0]);
    return rc;
  }
  const uint64_t n_total = n_bytes / block_size;
  std::vector<uint64_t> first(n), count(n);
  int T = 0;
  rc = cdx_plan_block_ranges(n_total, n, &T, first.data(), count.data());
  if (rc) return rc;
  rc = group_run(g, [&](int r) {
    return cdx_slot_commit_sharded_host(g->ctx[r], g->comm[r], count[r] ? data + first[r] * block_size : nullptr, count[r] * block_size, cell_size,
                                        block_size, first[r], n_total, T, &slots_out[r]);
  });
  if (rc) cdx_group_slots_free(g, slots_out);
  return rc;
}

extern "C" int cdx_group_slot_cell_paths(cdx_group* g, cdx_slot* const* slots, const uint64_t* cell_indices, size_t n_samples, size_t max_depth,
                                         uint8_t* out, uint8_t* leaf_out) {
  if (!g || !slots || !cell_indices || !out) return CDX_ERR_ARG;
  const size_t path_bytes = 32 * n_samples * max_depth, leaf_bytes = 32 * n_samples;
  return group_run(g, [&](int r) {
    std::vector<uint8_t> p(r == 0 ? 0 : path_bytes), l(r == 0 ? 0 : leaf_bytes);   // every rank receives the answer; rank 0's is returned
    return cdx_slot_cell_paths_sharded(slots[r], g->comm[r], cell_indices, n_samples, max_depth, r == 0 ? out : p.data(),
                                       r == 0 ? leaf_out : l.data());
  });
}

extern "C" void cdx_group_slots_free(cdx_group* g, cdx_slot** slots) {
  if (!g || !slots) return;
  for (size_t r = 0; r < g->ctx.size(); ++r) {
    cdx_slot_free(slots[r]);
    slots[r] = nullptr;
  }
}

extern "C" int cdx_group_dataset_commit(cdx_group* g, const cdx_slot_desc* slots, size_t n_slots, size_t cell_size, size_t block_size,
                                        int64_t keep_slot, cdx_dataset** datasets_out) {
  if (!g || !slots || !datasets_out) return CDX_ERR_ARG;
  for (size_t r = 0; r < g->ctx.size(); ++r) datasets_out[r] = nullptr;
  const int rc = group_run(g, [&](int r) { return cdx_dataset_commit(g->ctx[r], g->comm[r], slots, n_slots, cell_size, block_size, keep_slot, &datasets_out[r]); });
  if (rc) cdx_group_datasets_free(g, datasets_out);
  return rc;
}

extern "C" int cdx_group_dataset_prove(cdx_group* g, cdx_dataset* const* datasets, const uint8_t entropy[32], size_t n_samples, size_t max_depth,
                                       uint64_t* indices_out, uint8_t* paths_out, uint8_t* leaves_out) {
  if (!g || !datasets || !entropy || !indices_out || !paths_out) return CDX_ERR_ARG;
  return group_run(g, [&](int r) {
    std::vector<uint64_t> idx(r == 0 ? 0 : n_samples);
    std::vector<uint8_t> p(r == 0 ? 0 : 32 * n_samples * max_depth), l(r == 0 ? 0 : 32 * n_samples);
    return cdx_dataset_prove(datasets[r], entropy, n_samples, max_depth, r == 0 ? indices_out : idx.data(), r == 0 ? paths_out : p.data(),
                             r == 0 ? leaves_out : l.data());
  });
}

extern "C" void cdx_group_datasets_free(cdx_group* g, cdx_dataset** datasets) {
  if (!g || !datasets) return;
  for (size_t r = 0; r < g->ctx.size(); ++r) {
    cdx_dataset_free(datasets[r]);
    datasets[r] = nullptr;
  }
}
